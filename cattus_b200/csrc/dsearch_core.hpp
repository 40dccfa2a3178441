// Device-resident MCTS: the per-game steps of the reference's MctsPlayer (engine/src/mcts/mod.rs:105-454) written so
// that ONE WARP advances one game's search tree, with the tree in HBM.
//
// Why: the host driver (csrc/selfplay.cpp) runs the same search on host cores and is bound by them -- 4 cores per GPU on
// an 8-GPU box cannot feed an evaluator that does tens of millions of positions per second.  Here every game's trees live
// in device memory, `select` (mod.rs:199-244) is a warp-wide arg-max over a node's child rows, the leaf's bitboards are
// written STRAIGHT INTO THE EVALUATOR'S DEVICE RECORD BLOCK (no host round trip, no H2D copy), and create_children +
// backpropagate (mod.rs:246-281) consume the evaluator's device outputs.  One "wave" = begin (apply the host's per-move
// commands, tree reuse) -> select (all games) -> evaluator kernels -> expand (all games).
//
// What stays on the host (csrc/dsearch_host.hpp): everything that happens once per MOVE and draws random numbers -- the
// Dirichlet sample (double-precision libm: not bit-reproducible on the device), the temperature move choice, the game
// status, the .traindata entries.  A simulation never touches the host.
//
// Results are identical to the host driver's, game for game and byte for byte: the arithmetic of
// calc_selection_heuristic (mod.rs:233-244) is issued with round-to-nearest intrinsics in the reference's operation
// order (no FMA contraction), ties follow petgraph's newest-first edges() + max_by's last maximum (= smallest insertion
// index), tree reuse reverses child order as remove_all_but_subtree does, and the evaluator is batch invariant, so the
// ValueFuncCache of the host driver can simply be dropped (a hit returns what a fresh evaluation returns).
//
// The same source compiles for the host with a one-lane "warp" (DS_LANES == 1): tests/emul builds that into a
// test-only library which replays whole games against the host driver on CPU.  It is never part of the product library.
#pragma once

#include <cstdint>

#include "chess_rules.hpp"
#include "sp_rules.hpp"

namespace ds {

using sp::u128;

#if defined(__CUDA_ARCH__)
#define DS_DEVICE 1
#define DS_LANES 32
#else
#define DS_DEVICE 0
#define DS_LANES 1
#endif

// ------------------------------------------------------------------------------------------------ warp helpers
CB2_HD inline int lane() {
#if DS_DEVICE
    return static_cast<int>(threadIdx.x & 31u);
#else
    return 0;
#endif
}
CB2_HD inline void wsync() {
#if DS_DEVICE
    __syncwarp();
#endif
}
CB2_HD inline int wsum(int v) {
#if DS_DEVICE
    return __reduce_add_sync(0xFFFFFFFFu, v);
#else
    return v;
#endif
}
CB2_HD inline uint32_t wbcast(uint32_t v, int src = 0) {
#if DS_DEVICE
    return __shfl_sync(0xFFFFFFFFu, v, src);
#else
    (void)src;
    return v;
#endif
}
CB2_HD inline bool wany(bool p) {
#if DS_DEVICE
    return __any_sync(0xFFFFFFFFu, p) != 0;
#else
    return p;
#endif
}
// lowest lane whose predicate holds, or -1
CB2_HD inline int wfirst(bool p) {
#if DS_DEVICE
    const uint32_t m = __ballot_sync(0xFFFFFFFFu, p);
    return m ? __ffs(static_cast<int>(m)) - 1 : -1;
#else
    return p ? 0 : -1;
#endif
}
// (v, i) of the maximal v over the warp; equal values -> the smaller i
CB2_HD inline void wargmax(float& v, int& i, uint32_t& payload) {
#if DS_DEVICE
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const float ov = __shfl_xor_sync(0xFFFFFFFFu, v, d);
        const int oi = __shfl_xor_sync(0xFFFFFFFFu, i, d);
        const uint32_t op = __shfl_xor_sync(0xFFFFFFFFu, payload, d);
        if (ov > v || (ov == v && oi < i)) {
            v = ov;
            i = oi;
            payload = op;
        }
    }
#else
    (void)v;
    (void)i;
    (void)payload;
#endif
}
// exclusive prefix sum over the lanes; total = sum over the warp
CB2_HD inline int wexscan(int v, int& total) {
#if DS_DEVICE
    const int ln = static_cast<int>(threadIdx.x & 31u);
    int x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_up_sync(0xFFFFFFFFu, x, d);
        if (ln >= d) x += y;
    }
    total = __shfl_sync(0xFFFFFFFFu, x, 31);
    return x - v;
#else
    total = v;
    return 0;
#endif
}
CB2_HD inline uint32_t atomic_add_u32(uint32_t* p, uint32_t v) {
#if DS_DEVICE
    return atomicAdd(p, v);
#else
    const uint32_t o = *p;
    *p = o + v;
    return o;
#endif
}
CB2_HD inline void atomic_or_u32(uint32_t* p, uint32_t v) {
#if DS_DEVICE
    atomicOr(p, v);
#else
    *p |= v;
#endif
}
CB2_HD inline void atomic_add_u64(unsigned long long* p, unsigned long long v) {
#if DS_DEVICE
    atomicAdd(p, v);
#else
    *p += v;
#endif
}
// orders this thread's earlier writes to mapped host memory before its later ones, as the host sees them
CB2_HD inline void fence_system() {
#if DS_DEVICE
    __threadfence_system();
#else
    __atomic_thread_fence(__ATOMIC_SEQ_CST);
#endif
}
CB2_HD inline void atomic_max_u32(uint32_t* p, uint32_t v) {
#if DS_DEVICE
    atomicMax(p, v);
#else
    if (v > *p) *p = v;
#endif
}

// f32 operations of calc_selection_heuristic / add_dirichlet_noise / backpropagate, pinned to single IEEE operations so
// that nvcc cannot contract a multiply and an add into an FMA (the host driver is built with -ffp-contract=off)
CB2_HD inline float fmul(float a, float b) {
#if DS_DEVICE
    return __fmul_rn(a, b);
#else
    return a * b;
#endif
}
CB2_HD inline float fadd(float a, float b) {
#if DS_DEVICE
    return __fadd_rn(a, b);
#else
    return a + b;
#endif
}
CB2_HD inline float fdiv(float a, float b) {
#if DS_DEVICE
    return __fdiv_rn(a, b);
#else
    return a / b;
#endif
}
CB2_HD inline float fsqrt(float a) {
#if DS_DEVICE
    return __fsqrt_rn(a);
#else
    return __builtin_sqrtf(a);
#endif
}

// ------------------------------------------------------------------------------------------------ layouts
enum Phase : uint32_t { kIdle = 0, kRun = 1, kWaitEval = 2, kDone = 3 };
enum CmdFlags : uint32_t { kCmdNewGame = 1, kCmdMove = 2, kCmdStop = 4, kCmdSetRoot = 8, kCmdKeepTree = 16 };
enum ErrBits : uint32_t { kErrPool = 1, kErrPath = 2, kErrRows = 4, kErrNoise = 8 };

// One per concurrent game.  Scalars only; the per-slot arrays (tree pools, path, noise, history) are separate.
struct SlotState {
    uint32_t phase;  // Phase in the low 2 bits | (first wave in which select may run the slot) << 2: ONE word, because begin
                     // may run concurrently with the select of the same wave (begin_lead = 1)
    uint32_t cur, sims_left, pad0;
    int32_t root[2];
    uint32_t used[2];  // words in use of each player's tree pool
    uint32_t buf[2];   // which of the slot's three pool buffers holds each player's tree
    int32_t leaf;
    uint32_t row, path_len, noise_n;
    uint32_t hist_len, error, pad[2];
};

struct PathStep {
    int32_t c_idx;  // word index of the taken child's row {init, w, n, edge} in the tree's pool
    int32_t pad;
    int32_t child;  // block of the node the step leads to
};

// One child of a node: MctsEdge (mod.rs:32-45) + the link to the child's block.  16 bytes, so a lane fetches its child with
// ONE 128-bit load at an address that does not depend on the node's child count -- select issues it together with the
// header load, and the winner's edge word arrives with its score: one dependent global round trip per tree level.
struct alignas(16) Child {
    float init;     // init_score
    float w;        // score_w
    int32_t n;      // simulations_n
    uint32_t edge;  // (child block offset / 4 + 1) in the low 24 bits (0: not visited yet) | move << 24
};

// The evaluator's device-resident batch: [u32 n][pad to 16 B][record 0: 8-byte prefix | planes | legal bitmap] ...
struct EvalIo {
    uint32_t* n_ptr;      // rows in the batch (atomically allocated by select)
    uint8_t* recs;        // record 0's PLANES (the prefix [u32 prob offset][u32 #legal] sits 8 bytes before)
    const float* values;  // [max_rows]
    const float* probs;   // row r owns [r * prob_stride, r * prob_stride + #legal)
    uint32_t rec_bytes, prob_stride, max_rows, plane_words;
};

// ValueFuncCache (engine/src/mcts/cache.rs:31-75) in HBM: position key -> (probabilities over the legal moves in ascending
// nn index, value), exactly what the evaluator returned for it.  Set-associative: bucket = hash & mask, kCacheWays entries,
// first-in-first-out within a bucket.  A hit returns what a fresh evaluation would return (the evaluator is batch
// invariant), so games do not depend on the cache at all -- only the number of evaluator rows does.  Probes run in the
// select kernel, inserts in the expand kernel: the two never overlap, so only concurrent INSERTS need the bucket lock.
constexpr int kCacheWays = 4;
struct CacheIo {
    uint32_t* meta;    // per bucket 8 words: [lock][fifo cursor][tag x 4][pad x 2]; tag 0 = empty way
    uint8_t* entries;  // per entry: key 4 x u64 | u32 #legal | f32 value | f32 probs[max_children], padded to entry_bytes
    uint32_t bucket_mask, entry_bytes;
    uint32_t enabled, pad;
};

// Command block written by the host for one wave: [u32 n_cmds][u32 wave][8 B pad] then n_cmds commands of cmd_stride
// bytes: Cmd header + noise[max_children] f32.  kCmdSetRoot takes the slot's history from Params::roots[root_at, root_at +
// root_len) (oldest first, the root last).
struct Cmd {
    uint32_t slot, flags, move, cur, noise_n, root_at, root_len, pad;
};
// Result of one finished search, written by the device into mapped host memory: header + n[max_children] u32 +
// move[max_children] u16 (in insertion order; the host turns them into edges() order).  A search run in minibatches
// (batch_expand_slot) puts its minibatch and collision counts in pad[0] / pad[1]; the one-leaf kernels leave them unset.
struct ResultHdr {
    uint32_t slot, count, pad[2];
};
// Result of one finished search in analysis mode (Params::analysis): header + pv[kPvMax] u16 + n[max_children] u32 +
// w[max_children] f32 + init[max_children] f32 + move[max_children] u16, root children in insertion order.
constexpr uint32_t kPvMax = 16;
struct AnalysisHdr {
    uint32_t slot, count, pv_len, pad;
};

// One descent of a minibatch (Params::search_batch, DESIGN.md sections 15 and 16), written by batch_select_slot and
// backed up by batch_expand_slot.  Its path is Params::bpaths[slot][descent][0, depth).
enum DescentKind : uint32_t { kDescentCollision = 0, kDescentLeaf = 1, kDescentScored = 2 };
struct BatchDescent {
    int32_t leaf;    // block of the node the descent ended on
    uint32_t depth;  // edges on its path
    uint32_t kind;   // DescentKind
    uint32_t row;    // kDescentLeaf: the leaf's evaluator row
    float value;     // kDescentScored: repetition 0, finished position the winner's +-1 (player 1's view)
};

// Descents per minibatch of each side (indexed by SlotState::cur) and the larger of the two, which sizes each slot's
// descent records and paths.  Assigning one L gives both sides L (analysis searches one way throughout).
struct SearchBatch {
    uint32_t side[2];
    uint32_t max;
    CB2_HD SearchBatch& operator=(uint32_t L) {
        side[0] = side[1] = max = L;
        return *this;
    }
};

// A session (dsearch_session.hpp, DESIGN.md section 17) keeps one tree across searches.  Its control words live in mapped
// pinned memory: the host writes them, the device reads them in begin and at every minibatch boundary.
enum StopReason : uint32_t { kStopNone = 0, kStopNodes = 1, kStopMinibatches = 2, kStopRequest = 3, kStopDeadline = 4, kStopCapacity = 5 };
struct SessionCtl {
    uint32_t nodes;            // node budget of the search: new simulations on top of the kept tree (0xFFFFFFFF: none)
    uint32_t max_minibatches;  // minibatch cap (0xFFFFFFFF: none)
    uint32_t stop;             // kStopRequest / kStopDeadline: end at the next minibatch boundary
    uint32_t info;             // 1: post a snapshot after the next minibatch (the device clears it)
};
// A session's snapshot buffer: [u32 seq][u32 sims_done][u32 minibatches][u32 collisions] then one entry of the analysis
// result layout (result_stride bytes).  seq is odd while the device writes it; the last write is the even seq, behind a
// system-scope fence.
constexpr uint32_t kSnapshotHdr = 16;

template <class Rules>
struct Params {
    const void* rules;  // device copy of the rule tables (HexRulesT / ChessTables; unused for tic-tac-toe)
    SlotState* slots;
    uint32_t n_slots;
    uint32_t* pools;  // [n_slots][3][pool_words]
    uint32_t pool_words;
    PathStep* paths;  // [n_slots][path_cap]
    uint32_t path_cap;
    float* noise;  // [n_slots][max_children]
    uint32_t max_children;
    typename Rules::Pos* hist;  // [n_slots][hist_cap] ring; hist_cap is a power of two
    uint32_t hist_cap;
    EvalIo eval[2];
    CacheIo cache[2];
    uint32_t n_evals;
    uint32_t sim_num[2];
    float explore[2], noise_eps[2];
    const uint8_t* cmds;
    uint32_t cmd_stride;
    uint8_t* results;  // n_result_bufs buffers of result_buf_bytes; wave w uses buffer w % n_result_bufs
    uint32_t result_stride, n_result_bufs;
    unsigned long long result_buf_bytes;
    uint32_t* done_count;           // results posted in this wave (zeroed per wave)
    unsigned long long* counters;  // [0] simulations [1] evaluations [2] terminal leaves [3] cache hits
    uint32_t* error;                // sticky OR of ErrBits
    uint32_t* max_used;             // high-water mark of the words in use in any tree buffer (how close the pools came to full)
    uint32_t begin_lead;            // 0: begin runs before select in the same wave; 1: overlapped, effective next wave
    uint32_t visit_budget;          // node visits per slot and wave after which select stops starting new simulations
    uint32_t slot_base;             // the host's number of this population's slot 0 (two populations alternate waves)
    // analysis of given positions (dsearch_analysis.hpp); all zero in self-play
    const typename Rules::Pos* roots;  // root histories of this wave's kCmdSetRoot commands
    uint32_t analysis;                 // 1: finished searches post the AnalysisHdr layout instead of ResultHdr
    uint32_t pv_max;                   // principal variation plies to post (<= kPvMax)
    // minibatched search (batch_select_slot / batch_expand_slot); all zero with one leaf in flight
    SearchBatch search_batch;   // each side >= 1, max > 1
    BatchDescent* descents;     // [n_slots][search_batch.max]
    PathStep* bpaths;           // [n_slots][search_batch.max][path_cap]
    uint32_t* vcount;           // [n_slots][pool_words / 4]: virtual count of each child row (16-byte pool unit) of the tree
    // session (one slot searched in minibatches, begin_slot<true>); null outside sessions.  A session's sim_num is 0:
    // its budget is SessionCtl::nodes, and its begin resets the minibatch counts.
    volatile SessionCtl* session;
    uint8_t* snapshot;
};

template <class Pos>
struct alignas(16) NodeHdr {
    Pos pos;
    int32_t count;     // children (legal moves of pos; 0 for finished positions)
    int32_t expanded;  // rows are valid: create_children has run (mod.rs:246-262)
};

// Search tree storage: every visited node is one 16-byte-aligned block of 32-bit words
//   Header | Child[count] | move16[count] (chess)
// (the host driver keeps the four child fields as separate rows for its SIMD select; here a row per child suits a warp).
template <class Rules>
struct TreeOps {
    using Pos = typename Rules::Pos;
    using Hdr = NodeHdr<Pos>;
    static constexpr int kHdrWords = static_cast<int>((sizeof(Hdr) + 15) / 16 * 4);
    CB2_HD static Hdr* hdr(uint32_t* pool, int32_t b) { return reinterpret_cast<Hdr*>(pool + b); }
    CB2_HD static Child* child(uint32_t* pool, int32_t b) { return reinterpret_cast<Child*>(pool + b + kHdrWords); }
    CB2_HD static uint16_t* mv16(uint32_t* pool, int32_t b, int count) { return reinterpret_cast<uint16_t*>(pool + b + kHdrWords + 4 * count); }
    CB2_HD static uint32_t block_words(int count) {
        const uint32_t c = static_cast<uint32_t>(count);
        return (static_cast<uint32_t>(kHdrWords) + 4u * c + (Rules::kChess ? (c + 1u) / 2u : 0u) + 3u) & ~3u;
    }
    CB2_HD static uint32_t pack_edge(int32_t child_block, uint32_t m) {
        return (child_block < 0 ? 0u : (static_cast<uint32_t>(child_block >> 2) + 1u)) | (m << 24);
    }
    CB2_HD static int32_t edge_child(uint32_t e) { return (e & 0xFFFFFFu) ? static_cast<int32_t>(((e & 0xFFFFFFu) - 1u) << 2) : -1; }
    CB2_HD static uint32_t edge_move(uint32_t e) { return e >> 24; }
};

// The rule object a kernel works with: hex rules are a table struct read in place; chess rules wrap the table pointer.
template <class Rules>
struct RulesRef {
    CB2_HD static const Rules& get(const void* blob) { return *static_cast<const Rules*>(blob); }
};
template <>
struct RulesRef<sp::ChessRules> {
    CB2_HD static sp::ChessRules get(const void* blob) { return sp::ChessRules(*static_cast<const sp::ChessTables*>(blob)); }
};

template <class Rules>
struct Core {
    using Pos = typename Rules::Pos;
    using T = TreeOps<Rules>;
    using Hdr = typename T::Hdr;
    using P = Params<Rules>;
    static constexpr bool kChess = Rules::kChess;

    // registers of the tree a warp is working on (every lane holds the same copy; lane 0 stores them back)
    struct Tree {
        uint32_t* pool;
        uint32_t used;
        int32_t root;
    };

    CB2_HD static uint32_t move_at(uint32_t* pool, int32_t node, int count, int i) {
        if constexpr (kChess)
            return T::mv16(pool, node, count)[i];
        else
            return T::edge_move(T::child(pool, node)[i].edge);
    }

    // Appends the block of a node visited for the first time (rows zeroed, not expanded); -1 when the pool is full.
    // Its child count is the number of legal moves (0 for a finished position); for chess the moves themselves are
    // generated here, once, in the order NNetwork::evaluate returns them, and kept in the block.
    CB2_HD static int32_t add_node(const Rules& R, const P& p, Tree& t, const Pos& pos_in) {
        const int ln = lane();
        Pos pos = pos_in;
        int count = 0;
        if constexpr (kChess) {
            uint16_t buf[256];
            uint32_t packed = 0;
            if (ln == 0) {
                const int n = R.children(pos, buf);  // settles pos.st
                packed = static_cast<uint32_t>(n) | (static_cast<uint32_t>(pos.st) << 16);
            }
            packed = wbcast(packed);
            count = static_cast<int>(packed & 0xFFFFu);
            pos.st = static_cast<uint8_t>(packed >> 16);
            const uint32_t words = T::block_words(count);
            if (t.used + words > p.pool_words) return -1;
            const int32_t b = static_cast<int32_t>(t.used);
            t.used += words;
            if (ln == 0) {
                Hdr* h = T::hdr(t.pool, b);
                h->pos = pos;
                h->count = count;
                h->expanded = 0;
                uint16_t* mv = T::mv16(t.pool, b, count);
                for (int i = 0; i < count; ++i) mv[i] = buf[i];
            }
            Child* ch = T::child(t.pool, b);  // score_w and simulations_n start at zero, no child visited yet
            for (int i = ln; i < count; i += DS_LANES) ch[i] = Child{0.0f, 0.0f, 0, 0u};
            wsync();
            return b;
        } else {
            count = R.status(pos) != 0 ? 0 : sp::popcount128(R.legal_mask(pos));
            const uint32_t words = T::block_words(count);
            if (t.used + words > p.pool_words) return -1;
            const int32_t b = static_cast<int32_t>(t.used);
            t.used += words;
            if (ln == 0) {
                Hdr* h = T::hdr(t.pool, b);
                h->pos = pos;
                h->count = count;
                h->expanded = 0;
            }
            Child* ch = T::child(t.pool, b);
            for (int i = ln; i < count; i += DS_LANES) ch[i] = Child{0.0f, 0.0f, 0, 0u};
            wsync();
            return b;
        }
    }

    // First visit of child `i` of `node`: derive its position, append its block, link it.  -1 when the pool is full.
    CB2_HD static int32_t materialise(const Rules& R, const P& p, Tree& t, int32_t node, int count, int i) {
        const uint32_t m = move_at(t.pool, node, count, i);
        const Pos child = R.moved(T::hdr(t.pool, node)->pos, static_cast<typename Rules::Move>(m));
        const int32_t cb = add_node(R, p, t, child);
        if (cb < 0) return -1;
        if (lane() == 0) T::child(t.pool, node)[i].edge = T::pack_edge(cb, kChess ? 0u : m);
        wsync();
        return cb;
    }

    // mod.rs:270-281 along the recorded path; the side to move alternates from the root's
    CB2_HD static void backpropagate(uint32_t* pool, const PathStep* path, uint32_t depth, uint8_t root_turn, float score) {
        for (uint32_t j = static_cast<uint32_t>(lane()); j < depth; j += DS_LANES) {
            const uint8_t turn = (j & 1u) ? static_cast<uint8_t>(3 - root_turn) : root_turn;
            Child* c = reinterpret_cast<Child*>(pool + path[j].c_idx);
            c->n += 1;
            c->w = fadd(c->w, turn == 1 ? score : -score);
        }
    }

    // mod.rs:419-446 with the host's sample: zip(edges() order = newest first, noise)
    CB2_HD static void apply_noise(uint32_t* pool, int32_t node, int count, const float* nz, float eps) {
        Child* ch = T::child(pool, node);
        const float keep = 1.0f - eps;
        for (int i = lane(); i < count; i += DS_LANES) {
            float* x = &ch[count - 1 - i].init;
            *x = fadd(fmul(keep, *x), fmul(eps, nz[i]));
        }
    }

    // The finished search's root rows, for the host: calc_moves_probabilities' tail and the move choice run there.
    // Returns the posted entry.
    CB2_HD static uint8_t* post_results(const P& p, uint32_t wave, uint32_t si, uint32_t* pool, int32_t root) {
        if (p.analysis) return post_analysis(p, wave, si, pool, root);
        const int ln = lane();
        const int count = T::hdr(pool, root)->count;
        uint32_t k = 0;
        if (ln == 0) k = atomic_add_u32(p.done_count, 1u);
        k = wbcast(k);
        uint8_t* e = p.results + static_cast<unsigned long long>(wave % p.n_result_bufs) * p.result_buf_bytes + static_cast<size_t>(k) * p.result_stride;
        if (ln == 0) {
            ResultHdr* rh = reinterpret_cast<ResultHdr*>(e);
            rh->slot = si + p.slot_base;
            rh->count = static_cast<uint32_t>(count);
        }
        uint32_t* rn = reinterpret_cast<uint32_t*>(e + sizeof(ResultHdr));
        uint16_t* rm = reinterpret_cast<uint16_t*>(e + sizeof(ResultHdr) + 4u * p.max_children);
        const Child* ch = T::child(pool, root);
        for (int i = ln; i < count; i += DS_LANES) {
            rn[i] = static_cast<uint32_t>(ch[i].n);
            rm[i] = static_cast<uint16_t>(move_at(pool, root, count, i));
        }
        return e;
    }

    // Analysis result: every root row, and the principal variation -- from the root, repeatedly the child with the most
    // visits, equal counts going to the smallest insertion index (the last maximum in edges() order, as
    // choose_move_from_probabilities at temperature 0 picks), until a node that was never expanded or pv_max plies.
    // Returns the posted entry.
    CB2_HD static uint8_t* post_analysis(const P& p, uint32_t wave, uint32_t si, uint32_t* pool, int32_t root) {
        const int ln = lane();
        uint32_t k = 0;
        if (ln == 0) k = atomic_add_u32(p.done_count, 1u);
        k = wbcast(k);
        uint8_t* e = p.results + static_cast<unsigned long long>(wave % p.n_result_bufs) * p.result_buf_bytes + static_cast<size_t>(k) * p.result_stride;
        write_analysis(p, e, si, pool, root);
        return e;
    }

    // The analysis entry of the tree at `root`, written at `e`.
    CB2_HD static void write_analysis(const P& p, uint8_t* e, uint32_t si, uint32_t* pool, int32_t root) {
        const int ln = lane();
        const int count = T::hdr(pool, root)->count;
        uint16_t* pv = reinterpret_cast<uint16_t*>(e + sizeof(AnalysisHdr));
        uint32_t* rn = reinterpret_cast<uint32_t*>(e + sizeof(AnalysisHdr) + 2u * kPvMax);
        float* rw = reinterpret_cast<float*>(rn + p.max_children);
        float* ri = rw + p.max_children;
        uint16_t* rm = reinterpret_cast<uint16_t*>(ri + p.max_children);
        const Child* ch = T::child(pool, root);
        for (int i = ln; i < count; i += DS_LANES) {
            const Child c = ch[i];
            rn[i] = static_cast<uint32_t>(c.n);
            rw[i] = c.w;
            ri[i] = c.init;
            rm[i] = static_cast<uint16_t>(move_at(pool, root, count, i));
        }
        int32_t node = root;
        uint32_t len = 0;
        while (len < p.pv_max) {
            const Hdr* h = T::hdr(pool, node);
            const int cnt = h->count;
            if (!h->expanded || cnt == 0) break;
            const Child* c = T::child(pool, node);
            float bv = -1.0f;
            int bi = 0x7FFFFFFF;
            uint32_t be = 0;
            for (int i = ln; i < cnt; i += DS_LANES) {  // ascending i with a strict > keeps the smallest index among equals
                const float v = static_cast<float>(c[i].n);
                if (bi == 0x7FFFFFFF || v > bv) {
                    bv = v;
                    bi = i;
                    be = c[i].edge;
                }
            }
            wargmax(bv, bi, be);
            if (ln == 0) pv[len] = static_cast<uint16_t>(move_at(pool, node, cnt, bi));
            len += 1;
            node = T::edge_child(be);
            if (node < 0) break;
        }
        if (ln == 0) {
            AnalysisHdr* ah = reinterpret_cast<AnalysisHdr*>(e);
            ah->slot = si + p.slot_base;
            ah->count = static_cast<uint32_t>(count);
            ah->pv_len = len;
            ah->pad = 0;
        }
    }

    // MctsPlayer::detect_repetition (mod.rs:133-154), as the host driver does it: each path position is counted
    // against what precedes it; equal positions lie an even number of plies apart and not beyond the last pawn move or
    // capture (`rev`).  History older than hist_cap plies cannot matter (rev <= 101 under the fifty-move rule).
    CB2_HD static bool detect_repetition(const Rules&, const P& p, uint32_t* pool, const PathStep* path, uint32_t depth, uint32_t si,
                                         uint32_t hist_len) {
        if constexpr (!kChess) {
            return false;
        } else {
            const int32_t H = static_cast<int32_t>(hist_len);
            const Pos* hist = p.hist + static_cast<size_t>(si) * p.hist_cap;
            bool found = false;
            for (int32_t j = lane(); j < static_cast<int32_t>(depth) && !found; j += DS_LANES) {
                const Pos& a = T::hdr(pool, path[j].child)->pos;
                int seen = 1;
                for (int32_t d = 2; d <= a.rev; d += 2) {
                    const int32_t idx = H + j - d;
                    if (idx < 0) break;
                    const Pos& q = idx >= H ? T::hdr(pool, path[idx - H].child)->pos : hist[static_cast<uint32_t>(idx) & (p.hist_cap - 1u)];
                    if (Rules::same(a, q) && ++seen >= 3) {
                        found = true;
                        break;
                    }
                }
            }
            return wany(found);
        }
    }

    // NNetwork::evaluate's flip (net/mod.rs:74-87) + position_to_planes + legal moves, written as one evaluator record.
    // Returns the row, or 0xFFFFFFFF when the batch is full.
    CB2_HD static uint32_t emit_record(const Rules& R, const P& p, uint32_t e, uint32_t* pool, int32_t node) {
        const int ln = lane();
        const EvalIo& io = p.eval[e];
        uint32_t row = 0;
        if (ln == 0) row = atomic_add_u32(io.n_ptr, 1u);
        row = wbcast(row);
        if (row >= io.max_rows) return 0xFFFFFFFFu;
        uint8_t* rec = io.recs + static_cast<size_t>(row) * io.rec_bytes;
        const Hdr* h = T::hdr(pool, node);
        const int count = h->count;
        if constexpr (kChess) {
            uint32_t* bm = reinterpret_cast<uint32_t*>(rec + Rules::kPlanes * 8);
            const int bm_words = static_cast<int>((io.rec_bytes - 8u - Rules::kPlanes * 8u) / 4u);
            for (int i = ln; i < bm_words; i += DS_LANES) bm[i] = 0u;
            if (ln == 0) {
                uint64_t pl[Rules::kPlanes];
                R.planes(h->pos, pl);  // the stored position already is the evaluator's view
                uint64_t* out = reinterpret_cast<uint64_t*>(rec);
                for (int c = 0; c < Rules::kPlanes; ++c) out[c] = pl[c];
                uint32_t* prefix = reinterpret_cast<uint32_t*>(rec - 8);
                prefix[0] = row * io.prob_stride;
                prefix[1] = static_cast<uint32_t>(count);
            }
            wsync();
            const uint16_t* mv = T::mv16(pool, node, count);
            for (int i = ln; i < count; i += DS_LANES) {
                const int idx = R.nn_idx(mv[i]);
                atomic_or_u32(&bm[idx >> 5], 1u << (idx & 31));
            }
        } else {
            if (ln == 0) {
                const Pos ev = h->pos.turn != 1 ? R.flipped_boards(h->pos) : h->pos;
                u128 pl[3];
                R.planes(ev, pl);
                uint64_t* out = reinterpret_cast<uint64_t*>(rec);
                const int wpp = static_cast<int>(io.plane_words / 3u);
                for (int c = 0; c < 3; ++c)
                    for (int k = 0; k < wpp; ++k) out[c * wpp + k] = static_cast<uint64_t>(pl[c] >> (64 * k));
                uint32_t* prefix = reinterpret_cast<uint32_t*>(rec - 8);
                prefix[0] = row * io.prob_stride;
                prefix[1] = static_cast<uint32_t>(count);
            }
        }
        return row;
    }

    // ---------------------------------------------------------------------------------------- evaluation cache
    // The key of NNetwork::evaluate's cache lookup: the position as the network sees it (net/mod.rs:74-87).
    CB2_HD static uint64_t position_key(const Rules& R, const Pos& pos, uint64_t k[4]) {
        if constexpr (kChess) {
            R.key_planes(pos, k);
        } else {
            const Pos ev = pos.turn != 1 ? R.flipped_boards(pos) : pos;
            u128 pl[3];
            R.planes(ev, pl);
            k[0] = static_cast<uint64_t>(pl[0]);
            k[1] = static_cast<uint64_t>(pl[0] >> 64);
            k[2] = static_cast<uint64_t>(pl[1]);
            k[3] = static_cast<uint64_t>(pl[1] >> 64);
        }
        uint64_t h = 0x9E3779B97F4A7C15ull;
        for (int i = 0; i < 4; ++i) {
            uint64_t x = k[i] + 0x632BE59BD9B4E019ull * static_cast<uint64_t>(i + 1);
            x ^= x >> 33;
            x *= 0xff51afd7ed558ccdull;
            x ^= x >> 33;
            h = (h ^ x) * 0xc4ceb9fe1a85ec53ull;
        }
        return h ^ (h >> 29);
    }
    CB2_HD static uint32_t cache_tag(uint64_t h) {
        const uint32_t t = static_cast<uint32_t>(h >> 32);
        return t ? t : 1u;
    }
    // the entry holding `k`, or nullptr (uniform over the warp: every lane reads the same words)
    CB2_HD static const uint8_t* cache_find(const CacheIo& c, const uint64_t k[4], uint64_t h) {
        const uint32_t b = static_cast<uint32_t>(h) & c.bucket_mask;
        const uint32_t* meta = c.meta + static_cast<size_t>(b) * 8u;
        const uint32_t tag = cache_tag(h);
        for (int w = 0; w < kCacheWays; ++w) {
            if (meta[2 + w] != tag) continue;
            const uint8_t* e = c.entries + (static_cast<size_t>(b) * kCacheWays + static_cast<size_t>(w)) * c.entry_bytes;
            const uint64_t* ek = reinterpret_cast<const uint64_t*>(e);
            if (ek[0] == k[0] && ek[1] == k[1] && ek[2] == k[2] && ek[3] == k[3]) return e;
        }
        return nullptr;
    }
    // stores (probs[count], value) for `k` unless the key is already there (cache.rs:52-63)
    CB2_HD static void cache_insert(const CacheIo& c, const uint64_t k[4], uint64_t h, int count, const float* probs, float value) {
        const int ln = lane();
        const uint32_t b = static_cast<uint32_t>(h) & c.bucket_mask;
        uint32_t* meta = c.meta + static_cast<size_t>(b) * 8u;
        const uint32_t tag = cache_tag(h);
#if DS_DEVICE
        if (ln == 0) {
            while (atomicCAS(meta, 0u, 1u) != 0u) {
            }
            __threadfence();
        }
        __syncwarp();
#endif
        uint32_t way = 0xFFFFFFFFu;
        if (ln == 0) {
            bool present = false;
            for (int w = 0; w < kCacheWays; ++w) {
                const volatile uint32_t* vm = meta;
                if (vm[2 + w] == tag) {
                    const volatile uint64_t* ek = reinterpret_cast<const volatile uint64_t*>(c.entries + (static_cast<size_t>(b) * kCacheWays + static_cast<size_t>(w)) * c.entry_bytes);
                    if (ek[0] == k[0] && ek[1] == k[1] && ek[2] == k[2] && ek[3] == k[3]) present = true;
                }
            }
            if (!present) {
                const volatile uint32_t* vm = meta;
                for (int w = 0; w < kCacheWays && way == 0xFFFFFFFFu; ++w)
                    if (vm[2 + w] == 0u) way = static_cast<uint32_t>(w);
                if (way == 0xFFFFFFFFu) {  // bucket full: first in, first out within the bucket
                    way = vm[1] % static_cast<uint32_t>(kCacheWays);
                    meta[1] = way + 1u;
                }
            }
        }
        way = wbcast(way);
        if (way != 0xFFFFFFFFu) {
            uint8_t* e = c.entries + (static_cast<size_t>(b) * kCacheWays + way) * c.entry_bytes;
            float* ep = reinterpret_cast<float*>(e + 40);
            for (int i = ln; i < count; i += DS_LANES) ep[i] = probs[i];
            if (ln == 0) {
                uint64_t* ek = reinterpret_cast<uint64_t*>(e);
                ek[0] = k[0];
                ek[1] = k[1];
                ek[2] = k[2];
                ek[3] = k[3];
                *reinterpret_cast<uint32_t*>(e + 32) = static_cast<uint32_t>(count);
                *reinterpret_cast<float*>(e + 36) = value;
            }
        }
#if DS_DEVICE
        // entry, then tag, then one fence, then the unlock: the next holder of the lock (the only reader inside this kernel)
        // fences after acquiring it; select reads in a later kernel
        __syncwarp();
        if (ln == 0) {
            if (way != 0xFFFFFFFFu) meta[2 + way] = tag;
            __threadfence();
            atomicExch(meta, 0u);
        }
#else
        if (way != 0xFFFFFFFFu) meta[2 + way] = tag;
#endif
    }

    // create_children + root noise + backpropagate (mod.rs:180-194, :246-262) for `leaf` with the evaluator's answer for it
    // (fresh from the device batch, or from the cache): `probs` = calc_moves_probs' output, compact in ascending nn index.
    CB2_HD static void apply_evaluation(const Rules& R, const P& p, uint32_t si, uint32_t cur, uint32_t* pool, int32_t leaf, int32_t root,
                                        const float* probs, float value, uint32_t& noise_n, uint32_t depth) {
        const int ln = lane();
        Hdr* h = T::hdr(pool, leaf);
        const int count = h->count;
        const bool flipped = h->pos.turn != 1;
        Child* ch = T::child(pool, leaf);
        if constexpr (kChess) {
            // child i takes the entry at the rank of its nn index among the legal ones (net/mod.rs:106-119 gathers per
            // legal move); the edge row holds the nn indices while the ranks are counted, then becomes "no child yet"
            const uint16_t* mv = T::mv16(pool, leaf, count);
            for (int i = ln; i < count; i += DS_LANES) ch[i].edge = static_cast<uint32_t>(R.nn_idx(mv[i]));
            wsync();
            for (int i = ln; i < count; i += DS_LANES) {
                const uint32_t idx = ch[i].edge;
                int rank = 0;
                for (int j = 0; j < count; ++j) rank += ch[j].edge < idx ? 1 : 0;
                ch[i].init = probs[rank];
            }
            wsync();
            for (int i = ln; i < count; i += DS_LANES) ch[i].edge = T::pack_edge(-1, 0u);  // chess moves live in move16
        } else {
            // legal_moves() of the evaluated position, ascending; un-flipped by flip_score_if_needed (net/mod.rs:166-182)
            const Pos ev = flipped ? R.flipped_boards(h->pos) : h->pos;
            const u128 legal = R.legal_mask(ev);
            const int cells = R.moves_num();
            for (int cell = ln; cell < cells; cell += DS_LANES) {
                if (static_cast<uint32_t>(legal >> cell) & 1u) {
                    const int k = sp::popcount128(legal & (sp::bit128(cell) - 1));
                    ch[k].init = probs[k];
                    ch[k].edge = T::pack_edge(-1, static_cast<uint32_t>(flipped ? R.flip_move(cell) : cell));
                }
            }
        }
        if (ln == 0) h->expanded = 1;
        wsync();
        if (leaf == root && noise_n) {
            if (noise_n == static_cast<uint32_t>(count))
                apply_noise(pool, leaf, count, p.noise + static_cast<size_t>(si) * p.max_children, p.noise_eps[cur]);
            else if (ln == 0)
                atomic_or_u32(p.error, kErrNoise);
            noise_n = 0;
        }
        const float v = flipped ? -value : value;
        const uint8_t root_turn = T::hdr(pool, root)->pos.turn;
        backpropagate(pool, p.paths + static_cast<size_t>(si) * p.path_cap, depth, root_turn, v);
    }

    // ---------------------------------------------------------------------------------------- select (mod.rs:156-244)
    // Runs simulations of slot `si` until one needs the network (its record is written, the slot parks in kWaitEval) or
    // the search is out of simulations (results posted, kDone).  Terminal and repeated leaves are scored on the spot.
    CB2_HD static void select_slot(const Rules& R, const P& p, uint32_t si, uint32_t wave) {
        SlotState& S = p.slots[si];
        const uint32_t pw = S.phase;
        const uint32_t phase0 = pw & 3u, start_wave = pw >> 2;
        const uint32_t cur = S.cur;
        uint32_t sims_left = S.sims_left;
        Tree t;
        t.pool = p.pools + (static_cast<size_t>(si) * 3u + S.buf[cur & 1u]) * p.pool_words;
        t.used = S.used[cur & 1u];
        t.root = S.root[cur & 1u];
        const uint32_t hist_len = S.hist_len;
        uint32_t noise_n = S.noise_n;
        wsync();  // every lane holds its copy before lane 0 stores anything back
        if (phase0 != kRun || start_wave > wave) return;
        const int ln = lane();
        const uint32_t e = p.n_evals > 1 ? cur : 0u;
        PathStep* path = p.paths + static_cast<size_t>(si) * p.path_cap;
        const float ef = p.explore[cur];
        const uint8_t root_turn = T::hdr(t.pool, t.root)->pos.turn;
        uint32_t err = 0, phase = kRun, row = 0, path_len = 0, n_sims = 0, n_term = 0, n_hits = 0, visits = 0;
        const CacheIo& cache = p.cache[e];
        int32_t leaf = -1;
        for (;;) {
            if (sims_left == 0) {
                post_results(p, wave, si, t.pool, t.root);
                phase = kDone;
                break;
            }
            // Terminal and repeated leaves are scored on the spot and the slot goes on to its next simulation -- but only
            // within a budget of node visits per wave: near the end of a game nearly every simulation ends in a finished
            // position, and one warp walking hundreds of them would hold the whole wave (the kernel ends with its slowest
            // warp).  A slot over budget just sits this wave's batch out; its games are the same games.
            if (visits >= p.visit_budget) break;
            int32_t node = t.root;
            uint32_t depth = 0;
            for (;;) {
                const Hdr* h = T::hdr(t.pool, node);
                const Child* ch = T::child(t.pool, node);
                // this lane's first child, fetched BEFORE the child count is known (the address does not depend on it; a block
                // is followed by pool slack, so the read is in bounds even for a childless node) -- it travels with the header
                const Child c0 = ch[ln];
                const int count = h->count;
                if (!h->expanded || R.status(h->pos) != 0) break;
                int part = 0;
                for (int i = ln; i < count; i += DS_LANES) part += (i < DS_LANES ? c0.n : ch[i].n);
                const int simcount = 1 + wsum(part);
                const float sq = fsqrt(static_cast<float>(simcount));
                float bv = -__builtin_inff();
                int bi = 0x7FFFFFFF;
                uint32_t be = 0;
                for (int i = ln; i < count; i += DS_LANES) {
                    const Child c = i < DS_LANES ? c0 : ch[i];
                    const float exploit = c.n == 0 ? 0.0f : fdiv(c.w, static_cast<float>(c.n));
                    const float explore = fmul(fmul(ef, c.init), fdiv(sq, static_cast<float>(1 + c.n)));
                    const float v = fadd(exploit, explore);
                    // strict > over ascending i keeps the smallest index among equals; NaNs are never picked (the
                    // reference asserts them away, mod.rs:444)
                    if (v == v && (bi == 0x7FFFFFFF || v > bv)) {
                        bv = v;
                        bi = i;
                        be = c.edge;
                    }
                }
                wargmax(bv, bi, be);
                if (bi == 0x7FFFFFFF) {
                    bi = count - 1;
                    be = ch[bi].edge;
                }
                int32_t c = T::edge_child(be);
                if (c < 0) {
                    c = materialise(R, p, t, node, count, bi);
                    if (c < 0) {
                        err = kErrPool;
                        break;
                    }
                }
                if (depth >= p.path_cap) {
                    err = kErrPath;
                    break;
                }
                if (ln == 0) {
                    PathStep ps;
                    ps.c_idx = node + T::kHdrWords + 4 * bi;
                    ps.pad = 0;
                    ps.child = c;
                    path[depth] = ps;
                }
                depth += 1;
                node = c;
            }
            visits += depth + 1;
            if (err) break;
            wsync();  // the path is visible to every lane
            const Hdr* lh = T::hdr(t.pool, node);
            const bool repeated = detect_repetition(R, p, t.pool, path, depth, si, hist_len);
            const int st = R.status(lh->pos);
            if (repeated || st != 0) {
                const float v = repeated ? 0.0f : (st == 3 ? 0.0f : (st == 1 ? 1.0f : -1.0f));
                backpropagate(t.pool, path, depth, root_turn, v);
                sims_left -= 1;
                n_sims += 1;
                n_term += 1;
                wsync();
                continue;
            }
            if (cache.enabled) {  // ValueFuncCache::get_or_compute (cache.rs:31-75): a hit is expanded and scored on the spot
                uint64_t key[4];
                const uint64_t kh = position_key(R, lh->pos, key);
                const uint8_t* ce = cache_find(cache, key, kh);
                if (ce != nullptr && *reinterpret_cast<const uint32_t*>(ce + 32) == static_cast<uint32_t>(lh->count)) {
                    apply_evaluation(R, p, si, cur, t.pool, node, t.root, reinterpret_cast<const float*>(ce + 40), *reinterpret_cast<const float*>(ce + 36),
                                     noise_n, depth);
                    sims_left -= 1;
                    n_sims += 1;
                    n_hits += 1;
                    wsync();
                    continue;
                }
            }
            row = emit_record(R, p, e, t.pool, node);
            if (row == 0xFFFFFFFFu) {
                err = kErrRows;
                break;
            }
            leaf = node;
            path_len = depth;
            phase = kWaitEval;
            break;
        }
        if (ln == 0) {
            if (err) {
                atomic_or_u32(p.error, err);
                S.error = err;
                phase = kIdle;
            }
            S.phase = phase;
            S.sims_left = sims_left;
            S.used[cur & 1u] = t.used;
            if (t.used > S.pad0) {  // this slot's own high-water mark keeps the atomic off the common path
                S.pad0 = t.used;
                atomic_max_u32(p.max_used, t.used);
            }
            S.leaf = leaf;
            S.row = row;
            S.path_len = path_len;
            S.noise_n = noise_n;
            if (n_hits) atomic_add_u64(p.counters + 3, n_hits);
            if (n_sims) atomic_add_u64(p.counters + 0, n_sims);
            if (n_term) atomic_add_u64(p.counters + 2, n_term);
            if (phase == kWaitEval) atomic_add_u64(p.counters + 1, 1ull);
        }
    }

    // ------------------------------------------------- create_children + root noise + backpropagate (mod.rs:180-194)
    CB2_HD static void expand_slot(const Rules& R, const P& p, uint32_t si, uint32_t wave) {
        SlotState& S = p.slots[si];
        const uint32_t phase0 = S.phase & 3u, cur = S.cur, row = S.row, depth = S.path_len;
        uint32_t sims_left = S.sims_left, noise_n = S.noise_n;
        const int32_t leaf = S.leaf;
        uint32_t* pool = p.pools + (static_cast<size_t>(si) * 3u + S.buf[cur & 1u]) * p.pool_words;
        const int32_t root = S.root[cur & 1u];
        wsync();
        if (phase0 != kWaitEval) return;
        const int ln = lane();
        const uint32_t e = p.n_evals > 1 ? cur : 0u;
        const EvalIo& io = p.eval[e];
        const float* probs = io.probs + static_cast<size_t>(row) * io.prob_stride;
        const float value = io.values[row];
        if (p.cache[e].enabled) {
            uint64_t key[4];
            const uint64_t kh = position_key(R, T::hdr(pool, leaf)->pos, key);
            cache_insert(p.cache[e], key, kh, T::hdr(pool, leaf)->count, probs, value);
        }
        apply_evaluation(R, p, si, cur, pool, leaf, root, probs, value, noise_n, depth);
        sims_left -= 1;
        uint32_t phase = kRun;
        if (sims_left == 0) {
            wsync();
            post_results(p, wave, si, pool, root);
            phase = kDone;
        }
        if (ln == 0) {
            S.phase = phase;
            S.sims_left = sims_left;
            S.noise_n = noise_n;
            atomic_add_u64(p.counters + 0, 1ull);
        }
    }

    // ---------------------------------------------------------------- minibatches under virtual loss (DESIGN.md section 15)
    // Any search with search_batch[cur] = L (analysis, and self-play / match play when a side has L > 1; a side with
    // L = 1 gets develop_tree's result).  One wave runs one minibatch of a slot: batch_select_slot makes its
    // k = min(L, sims_left) descents, batch_expand_slot backs them up once the evaluator has run.  The slot keeps
    // the number of descents in flight in path_len and its minibatch / collision counts in pad[0] / pad[1].
    //
    // Phase 1: descents j = 0 .. k-1 in order on a FROZEN tree (no n, w or children change; first visits of an edge are
    // linked as select links them).  Every child row is seen with its virtual count v, the descents of this minibatch
    // that took it so far: n' = n + v, w' = w - v, then select's heuristic and tie rule; with every v = 0 this is select
    // bit for bit.  A descent ends where select ends and is a repetition (value 0), a finished position (the winner's
    // +-1), a new leaf (the first to end on that unexpanded node: claimed with expanded = 2, its record written to the
    // evaluator batch) or a collision (a later one), then adds 1 to v along its path.  No cache probe: a hit would have
    // to be copied out before the expand kernel's inserts could evict it, and the tree's own leaves fill the batch.
    CB2_HD static void batch_select_slot(const Rules& R, const P& p, uint32_t si, uint32_t wave) {
        SlotState& S = p.slots[si];
        const uint32_t pw = S.phase;
        const uint32_t phase0 = pw & 3u, start_wave = pw >> 2;
        const uint32_t cur = S.cur;
        const uint32_t sims_left = S.sims_left;
        Tree t;
        t.pool = p.pools + (static_cast<size_t>(si) * 3u + S.buf[cur & 1u]) * p.pool_words;
        t.used = S.used[cur & 1u];
        t.root = S.root[cur & 1u];
        const uint32_t hist_len = S.hist_len;
        wsync();
        if (phase0 != kRun || start_wave > wave) return;
        const int ln = lane();
        const uint32_t e = p.n_evals > 1 ? cur : 0u;
        const float ef = p.explore[cur];
        const uint32_t L = (cur & 1u) ? p.search_batch.side[1] : p.search_batch.side[0];
        const uint32_t stride = p.search_batch.max;
        const uint32_t k = sims_left < L ? sims_left : L;
        uint32_t* vc = p.vcount + static_cast<size_t>(si) * (p.pool_words >> 2);
        BatchDescent* bd = p.descents + static_cast<size_t>(si) * stride;
        uint32_t err = 0, rows = 0;
        for (uint32_t j = 0; j < k && !err; ++j) {
            PathStep* path = p.bpaths + (static_cast<size_t>(si) * stride + j) * p.path_cap;
            int32_t node = t.root;
            uint32_t depth = 0;
            for (;;) {
                const Hdr* h = T::hdr(t.pool, node);
                if (h->expanded != 1 || R.status(h->pos) != 0) break;
                const int count = h->count;
                const Child* ch = T::child(t.pool, node);
                const uint32_t* vn = vc + ((static_cast<uint32_t>(node) + T::kHdrWords) >> 2);
                int part = 0;
                for (int i = ln; i < count; i += DS_LANES) part += ch[i].n + static_cast<int>(vn[i]);
                const int simcount = 1 + wsum(part);
                const float sq = fsqrt(static_cast<float>(simcount));
                float bv = -__builtin_inff();
                int bi = 0x7FFFFFFF;
                uint32_t be = 0;
                for (int i = ln; i < count; i += DS_LANES) {
                    const Child c = ch[i];
                    const uint32_t v = vn[i];
                    const int n = c.n + static_cast<int>(v);
                    const float w = fadd(c.w, -static_cast<float>(v));
                    const float exploit = n == 0 ? 0.0f : fdiv(w, static_cast<float>(n));
                    const float explore = fmul(fmul(ef, c.init), fdiv(sq, static_cast<float>(1 + n)));
                    const float s = fadd(exploit, explore);
                    if (s == s && (bi == 0x7FFFFFFF || s > bv)) {
                        bv = s;
                        bi = i;
                        be = c.edge;
                    }
                }
                wargmax(bv, bi, be);
                if (bi == 0x7FFFFFFF) {
                    bi = count - 1;
                    be = ch[bi].edge;
                }
                int32_t c = T::edge_child(be);
                if (c < 0) {
                    c = materialise(R, p, t, node, count, bi);
                    if (c < 0) {
                        err = kErrPool;
                        break;
                    }
                }
                if (depth >= p.path_cap) {
                    err = kErrPath;
                    break;
                }
                if (ln == 0) {
                    PathStep ps;
                    ps.c_idx = node + T::kHdrWords + 4 * bi;
                    ps.pad = 0;
                    ps.child = c;
                    path[depth] = ps;
                }
                depth += 1;
                node = c;
            }
            if (err) break;
            wsync();
            Hdr* lh = T::hdr(t.pool, node);
            BatchDescent d;
            d.leaf = node;
            d.depth = depth;
            d.row = 0;
            d.value = 0.0f;
            const bool repeated = detect_repetition(R, p, t.pool, path, depth, si, hist_len);
            const int st = R.status(lh->pos);
            if (repeated || st != 0) {
                d.kind = kDescentScored;
                d.value = repeated ? 0.0f : (st == 3 ? 0.0f : (st == 1 ? 1.0f : -1.0f));
            } else if (lh->expanded == 2) {
                d.kind = kDescentCollision;
            } else {
                d.kind = kDescentLeaf;
                d.row = emit_record(R, p, e, t.pool, node);
                if (d.row == 0xFFFFFFFFu) {
                    err = kErrRows;
                    break;
                }
                rows += 1;
                if (ln == 0) lh->expanded = 2;
            }
            for (uint32_t s = static_cast<uint32_t>(ln); s < depth; s += DS_LANES) vc[static_cast<uint32_t>(path[s].c_idx) >> 2] += 1u;
            if (ln == 0) bd[j] = d;
            wsync();
        }
        if (ln == 0) {  // the slot's scalars are read again rather than kept live across the descents
            SlotState& Q = p.slots[si];
            const uint32_t qc = Q.cur, left = Q.sims_left;
            uint32_t phase = kWaitEval;
            if (err) {
                atomic_or_u32(p.error, err);
                Q.error = err;
                phase = kIdle;
            }
            Q.phase = phase;
            const uint32_t L = (qc & 1u) ? p.search_batch.side[1] : p.search_batch.side[0];
            Q.path_len = left < L ? left : L;
            Q.used[qc & 1u] = t.used;
            if (t.used > Q.pad0) {
                Q.pad0 = t.used;
                atomic_max_u32(p.max_used, t.used);
            }
            if (left == p.sim_num[qc]) {  // the search's first minibatch
                Q.pad[0] = 0;
                Q.pad[1] = 0;
            }
            if (rows) atomic_add_u64(p.counters + 1, rows);
        }
    }

    // Phase 3: in descent order, a new leaf gets create_children from its evaluation, then it and every scored descent is
    // backpropagated as expand_slot / select do; a collision does nothing.  Per edge that is a sum in ascending descent
    // order, as the sequential definition adds.  Then every virtual count of the minibatch is dropped.  A root that a
    // minibatch expands takes the host's noise sample as expand_slot's does.
    CB2_HD static void batch_expand_slot(const Rules& R, const P& p, uint32_t si, uint32_t wave) {
        SlotState& S = p.slots[si];
        const uint32_t phase0 = S.phase & 3u, cur = S.cur, k = S.path_len;
        uint32_t* pool = p.pools + (static_cast<size_t>(si) * 3u + S.buf[cur & 1u]) * p.pool_words;
        const int32_t root = S.root[cur & 1u];
        wsync();
        if (phase0 != kWaitEval) return;
        const int ln = lane();
        const uint32_t e = p.n_evals > 1 ? cur : 0u;
        const EvalIo& io = p.eval[e];
        const uint32_t stride = p.search_batch.max;
        const uint8_t root_turn = T::hdr(pool, root)->pos.turn;
        uint32_t* vc = p.vcount + static_cast<size_t>(si) * (p.pool_words >> 2);
        const BatchDescent* bd = p.descents + static_cast<size_t>(si) * stride;
        uint32_t n_sims = 0, n_scored = 0, n_coll = 0;
        for (uint32_t j = 0; j < k; ++j) {
            const BatchDescent d = bd[j];
            const PathStep* path = p.bpaths + (static_cast<size_t>(si) * stride + j) * p.path_cap;
            if (d.kind == kDescentCollision) {
                n_coll += 1;
                continue;
            }
            float v = d.value;
            if (d.kind == kDescentLeaf) {
                const float* probs = io.probs + static_cast<size_t>(d.row) * io.prob_stride;
                const float value = io.values[d.row];
                if (p.cache[e].enabled) {
                    uint64_t key[4];
                    const uint64_t kh = position_key(R, T::hdr(pool, d.leaf)->pos, key);
                    cache_insert(p.cache[e], key, kh, T::hdr(pool, d.leaf)->count, probs, value);
                }
                // the root's noise count is read only where a minibatch expands the root, rather than kept live
                uint32_t noise_n = d.leaf == root ? p.slots[si].noise_n : 0u;
                wsync();
                apply_evaluation(R, p, si, cur, pool, d.leaf, root, probs, value, noise_n, 0u);  // children only: depth 0
                if (d.leaf == root && ln == 0) p.slots[si].noise_n = noise_n;
                v = T::hdr(pool, d.leaf)->pos.turn != 1 ? -value : value;
            } else {
                n_scored += 1;
            }
            wsync();
            backpropagate(pool, path, d.depth, root_turn, v);
            n_sims += 1;
            wsync();
        }
        for (uint32_t j = 0; j < k; ++j) {
            const uint32_t depth = bd[j].depth;
            const PathStep* path = p.bpaths + (static_cast<size_t>(si) * stride + j) * p.path_cap;
            for (uint32_t s = static_cast<uint32_t>(ln); s < depth; s += DS_LANES) vc[static_cast<uint32_t>(path[s].c_idx) >> 2] = 0u;
        }
        wsync();
        // the slot's counts are read here rather than kept live across the backups
        SlotState& Q = p.slots[si];
        const uint32_t left = Q.sims_left - n_sims, minibatches = Q.pad[0] + 1u, collisions = Q.pad[1] + n_coll;
        wsync();
        uint32_t phase = kRun;
        uint32_t reason = left == 0 ? kStopNodes : kStopNone;
        // the host writes the session's words at any time: lane 0 reads them and the warp takes its decision
        if (p.session && reason == kStopNone) reason = wbcast(ln == 0 ? session_stop(p, Q.used[cur & 1u], minibatches) : 0u);
        if (reason != kStopNone) {
            uint8_t* entry = post_results(p, wave, si, pool, root);
            if (ln == 0) {  // the analysis entry ends in the two counts; the self-play one has them in ResultHdr::pad
                uint32_t* counts = p.analysis ? reinterpret_cast<uint32_t*>(entry + p.result_stride - 16u) : reinterpret_cast<ResultHdr*>(entry)->pad;
                counts[0] = minibatches;
                counts[1] = collisions;
                if (p.session) {  // a session's entry also carries the visits the search kept and why it ended
                    counts[2] = Q.row;
                    counts[3] = reason;
                }
            }
            phase = kDone;
        }
        if (p.session && (reason != kStopNone || wbcast(ln == 0 ? p.session->info : 0u) != 0u)) post_snapshot(p, si, pool, root, left, minibatches, collisions);
        if (ln == 0) {
            Q.phase = phase;
            Q.sims_left = left;
            Q.pad[0] = minibatches;
            Q.pad[1] = collisions;
            if (n_sims) atomic_add_u64(p.counters + 0, n_sims);
            if (n_scored) atomic_add_u64(p.counters + 2, n_scored);
        }
    }

    // Why a session's search ends at this minibatch boundary besides its node budget (kStopNone: it goes on): the minibatch
    // cap, a stop or deadline the host wrote, or a tree buffer that might not hold another minibatch's new leaves.
    CB2_HD static uint32_t session_stop(const P& p, uint32_t used, uint32_t minibatches) {
        if (minibatches >= p.session->max_minibatches) return kStopMinibatches;
        const uint32_t stop = p.session->stop;
        if (stop != kStopNone) return stop;
        if (static_cast<unsigned long long>(used) + minibatch_words(p) > p.pool_words) return kStopCapacity;
        return kStopNone;
    }
    // the most a minibatch can add to a tree: each descent materialises at most one node
    CB2_HD static unsigned long long minibatch_words(const P& p) {
        return static_cast<unsigned long long>(p.search_batch.max) * T::block_words(static_cast<int>(p.max_children));
    }

    // The session's snapshot: the analysis entry of the tree as it stands, with the search's counts, behind a sequence
    // word the host checks before and after it reads.
    CB2_HD static void post_snapshot(const P& p, uint32_t si, uint32_t* pool, int32_t root, uint32_t left, uint32_t minibatches, uint32_t collisions) {
        const int ln = lane();
        volatile uint32_t* hdr = reinterpret_cast<volatile uint32_t*>(p.snapshot);
        const uint32_t seq = wbcast(ln == 0 ? hdr[0] : 0u) | 1u;
        if (ln == 0) hdr[0] = seq;
        fence_system();
        wsync();
        write_analysis(p, p.snapshot + kSnapshotHdr, si, pool, root);
        if (ln == 0) {
            hdr[1] = p.session->nodes - left;
            hdr[2] = minibatches;
            hdr[3] = collisions;
        }
        wsync();
        fence_system();
        if (ln == 0) {
            hdr[0] = seq + 1u;
            p.session->info = 0;
        }
    }

    // ------------------------------------------------------------------ tree reuse (mod.rs:283-352)
    CB2_HD static bool child_matches(const Rules& R, const Pos& parent, uint32_t m, const Pos& target) {
        if constexpr (kChess) {
            if (target.turn != 3 - parent.turn) return false;
            // cheap necessary conditions before the full make-move: in the target (the opponent's view, ranks
            // mirrored) the origin square is empty and the destination holds a piece of the side that just moved
            const int from = Rules::from_of(static_cast<uint16_t>(m)) ^ 56, to = Rules::to_of(static_cast<uint16_t>(m)) ^ 56;
            const uint64_t all = Rules::occ(target);
            if ((all >> from) & 1ull) return false;
            if (!(((all & ~target.us) >> to) & 1ull)) return false;
            return Rules::same(R.moved(parent, static_cast<uint16_t>(m)), target);
        } else {
            return R.child_matches(parent, static_cast<int>(m), target);
        }
    }

    // one BFS node of find_node_with_position: its children in edges() order (newest first); returns the matching child's
    // block (materialised if it had none), -1 for no match, -2 when the pool is full
    CB2_HD static int32_t scan_children(const Rules& R, const P& p, Tree& t, int32_t node, const Pos& position) {
        const Hdr* h = T::hdr(t.pool, node);
        if (!h->expanded) return -1;
        const int count = h->count;
        const Child* ch = T::child(t.pool, node);
        for (int base = 0; base < count; base += DS_LANES) {
            const int i = count - 1 - (base + lane());
            bool hit = false;
            if (i >= 0) {
                const int32_t c = T::edge_child(ch[i].edge);
                if (c >= 0)
                    hit = R.same(T::hdr(t.pool, c)->pos, position);
                else
                    hit = child_matches(R, h->pos, move_at(t.pool, node, count, i), position);
            }
            const int f = wfirst(hit);
            if (f >= 0) {
                const int fi = count - 1 - (base + f);
                int32_t c = T::edge_child(ch[fi].edge);
                if (c < 0) {
                    c = materialise(R, p, t, node, count, fi);
                    if (c < 0) return -2;
                }
                return c;
            }
        }
        return -1;
    }

    // mod.rs:283-301, depth_limit = 3 (root, its children, their children)
    CB2_HD static int32_t find_node_with_position(const Rules& R, const P& p, Tree& t, const Pos& position) {
        if (R.same(T::hdr(t.pool, t.root)->pos, position)) return t.root;
        int32_t r = scan_children(R, p, t, t.root, position);
        if (r != -1) return r;
        const Hdr* rh = T::hdr(t.pool, t.root);
        if (!rh->expanded) return -1;
        const int count = rh->count;
        for (int i = count - 1; i >= 0; --i) {
            const int32_t c = T::edge_child(T::child(t.pool, t.root)[i].edge);
            if (c < 0) continue;
            r = scan_children(R, p, t, c, position);
            if (r != -1) return r;
        }
        return -1;
    }

    // mod.rs:303-333: the subtree is copied into the slot's spare buffer; edges are re-inserted in iteration
    // (newest-first) order, so every kept node's child order is reversed.  The copy is breadth-first with ONE NODE PER
    // LANE: a queue of (new block, old block) pairs grows down from the top of the new pool while the blocks grow up
    // from its bottom; each round the lanes take up to 32 queued nodes, size their visited children (pass 1), get their
    // block and queue ranges from two warp scans, then copy their rows reversed and enqueue the children (pass 2).
    // A node-serial copy made tree reuse the bottleneck of whole games: ~2 us of dependent loads per kept node.
    // Block offsets differ from the host driver's depth-first copy; nothing observable depends on them.
    CB2_HD static bool copy_subtree(const P& p, const uint32_t* old_pool_c, int32_t sub_root, Tree& nt) {
        uint32_t* old_pool = const_cast<uint32_t*>(old_pool_c);
        const int ln = lane();
        uint32_t* q = nt.pool + p.pool_words;  // entry e lives in q[-2 (e + 1)], q[-2 (e + 1) + 1]
        {
            const Hdr* oh = T::hdr(old_pool, sub_root);
            const uint32_t words = T::block_words(oh->count);
            if (words + 2u > p.pool_words) return false;
            if (ln == 0) {
                Hdr* nh = T::hdr(nt.pool, 0);
                nh->pos = oh->pos;
                nh->count = oh->count;
                nh->expanded = 0;
                q[-2] = 0u;
                q[-1] = static_cast<uint32_t>(sub_root);
            }
            nt.used = words;
            nt.root = 0;
        }
        uint32_t q_head = 0, q_tail = 1;
        wsync();
        while (q_head < q_tail) {
            const uint32_t e = q_head + static_cast<uint32_t>(ln);
            const bool active = e < q_tail;
            int32_t nb = 0, ob = 0;
            int count = 0, need = 0, kids = 0;
            bool expanded = false;
            if (active) {
                nb = static_cast<int32_t>(q[-2 * static_cast<int32_t>(e + 1u)]);
                ob = static_cast<int32_t>(q[-2 * static_cast<int32_t>(e + 1u) + 1]);
                const Hdr* oh = T::hdr(old_pool, ob);
                count = oh->count;
                expanded = oh->expanded != 0;
                if (expanded) {
                    const Child* och = T::child(old_pool, ob);
                    for (int o = 0; o < count; ++o) {
                        const int32_t oc = T::edge_child(och[o].edge);
                        if (oc >= 0) {
                            need += static_cast<int>(T::block_words(T::hdr(old_pool, oc)->count));
                            kids += 1;
                        }
                    }
                }
            }
            int total_need = 0, total_kids = 0;
            const int off = wexscan(need, total_need);
            const int koff = wexscan(kids, total_kids);
            // blocks grow up, the queue grows down: they must not meet
            if (static_cast<unsigned long long>(nt.used) + static_cast<uint32_t>(total_need) + 2ull * (q_tail + static_cast<uint32_t>(total_kids)) > p.pool_words)
                return false;
            if (active) {
                Hdr* nh = T::hdr(nt.pool, nb);
                if (!expanded) {
                    // visited but never expanded: no edges yet, nothing to reverse -- chess moves keep their generated order
                    Child* nch = T::child(nt.pool, nb);
                    for (int i = 0; i < count; ++i) nch[i] = Child{0.0f, 0.0f, 0, 0u};
                    if constexpr (kChess) {
                        const uint16_t* om = T::mv16(old_pool, ob, count);
                        uint16_t* nm = T::mv16(nt.pool, nb, count);
                        for (int i = 0; i < count; ++i) nm[i] = om[i];
                    }
                    nh->expanded = 0;
                } else {
                    const Child* och = T::child(old_pool, ob);
                    Child* nch = T::child(nt.pool, nb);
                    uint32_t next_block = nt.used + static_cast<uint32_t>(off);
                    uint32_t next_q = q_tail + static_cast<uint32_t>(koff);
                    for (int i = 0; i < count; ++i) {  // new insertion order = old iteration order (newest first)
                        const int o = count - 1 - i;
                        Child c = och[o];
                        if constexpr (kChess) T::mv16(nt.pool, nb, count)[i] = T::mv16(old_pool, ob, count)[o];
                        const int32_t oc = T::edge_child(c.edge);
                        int32_t nc = -1;
                        if (oc >= 0) {
                            const Hdr* ohc = T::hdr(old_pool, oc);
                            nc = static_cast<int32_t>(next_block);
                            next_block += T::block_words(ohc->count);
                            Hdr* chd = T::hdr(nt.pool, nc);
                            chd->pos = ohc->pos;
                            chd->count = ohc->count;
                            chd->expanded = 0;
                            q[-2 * static_cast<int32_t>(next_q + 1u)] = static_cast<uint32_t>(nc);
                            q[-2 * static_cast<int32_t>(next_q + 1u) + 1] = static_cast<uint32_t>(oc);
                            next_q += 1;
                        }
                        c.edge = T::pack_edge(nc, T::edge_move(c.edge));
                        nch[i] = c;
                    }
                    nh->expanded = 1;
                }
            }
            const uint32_t batch = q_tail - q_head < static_cast<uint32_t>(DS_LANES) ? q_tail - q_head : static_cast<uint32_t>(DS_LANES);
            nt.used += static_cast<uint32_t>(total_need);
            q_tail += static_cast<uint32_t>(total_kids);
            q_head += batch;
            wsync();
        }
        return true;
    }

    // One host command: optional new game / move, then calc_moves_probabilities up to develop_tree (mod.rs:335-362) for
    // the player `cur`: find the position in the kept tree, keep its subtree, else start from a fresh root.
    // kSession (a session's begin, DESIGN.md section 17): kCmdSetRoot | kCmdKeepTree installs the history but looks for its
    // last position in the kept tree; a kept tree that cannot be copied, or has no room for one more minibatch, gives way
    // to a fresh root; the budget is SessionCtl::nodes, and the slot records the root's visits before the search in `row`.
    template <bool kSession = false>
    CB2_HD static void begin_slot(const Rules& R, const P& p, uint32_t ci, uint32_t wave) {
        const uint8_t* cb = p.cmds + 16 + static_cast<size_t>(ci) * p.cmd_stride;
        const Cmd cmd = *reinterpret_cast<const Cmd*>(cb);
        const float* cmd_noise = reinterpret_cast<const float*>(cb + sizeof(Cmd));
        const uint32_t si = cmd.slot - p.slot_base;
        if (si >= p.n_slots) return;
        SlotState& S = p.slots[si];
        int32_t root[2] = {S.root[0], S.root[1]};
        uint32_t used[2] = {S.used[0], S.used[1]};
        uint32_t buf[2] = {S.buf[0], S.buf[1]};
        uint32_t hist_len = S.hist_len;
        wsync();
        const int ln = lane();
        if (cmd.flags & kCmdStop) {
            if (ln == 0) S.phase = kIdle;
            return;
        }
        Pos* hist = p.hist + static_cast<size_t>(si) * p.hist_cap;
        const uint32_t hmask = p.hist_cap - 1u;
        if (cmd.flags & kCmdNewGame) {
            root[0] = root[1] = -1;
            used[0] = used[1] = 0;
            buf[0] = 0;
            buf[1] = 1;
            hist_len = 1;
            if (ln == 0) hist[0] = R.initial();
        } else if (cmd.flags & kCmdSetRoot) {
            // a fresh tree at a position the host gives, with the history detect_repetition looks back into
            if (!kSession || !(cmd.flags & kCmdKeepTree)) {
                root[0] = root[1] = -1;
                used[0] = used[1] = 0;
                buf[0] = 0;
                buf[1] = 1;
            }
            hist_len = cmd.root_len;
            for (uint32_t i = static_cast<uint32_t>(ln); i < hist_len; i += DS_LANES) hist[i] = p.roots[cmd.root_at + i];
        } else if (cmd.flags & kCmdMove) {
            if (ln == 0) {
                Pos np = R.moved(hist[(hist_len - 1u) & hmask], static_cast<typename Rules::Move>(cmd.move));
                if constexpr (kChess) {
                    uint16_t mbuf[256];
                    R.children(np, mbuf);  // settles status()
                }
                hist[hist_len & hmask] = np;
            }
            hist_len += 1;
        }
        wsync();
        const Pos position = hist[(hist_len - 1u) & hmask];
        const uint32_t cur = cmd.cur & 1u;
        Tree t;
        t.pool = p.pools + (static_cast<size_t>(si) * 3u + buf[cur]) * p.pool_words;
        t.used = used[cur];
        t.root = root[cur];
        uint32_t err = 0;
        bool reused = false;
        if (t.root >= 0) {
            const int32_t node = find_node_with_position(R, p, t, position);
            if (node == -2 && !kSession) {
                err = kErrPool;
            } else if (node >= 0) {
                if (node != t.root) {
                    Tree nt;
                    const uint32_t spare = 3u - buf[0] - buf[1];
                    nt.pool = p.pools + (static_cast<size_t>(si) * 3u + spare) * p.pool_words;
                    nt.used = 0;
                    nt.root = 0;
                    if (copy_subtree(p, t.pool, node, nt)) {
                        buf[cur] = spare;
                        t = nt;
                        reused = true;
                    } else if (kSession) {
                        t.root = -1;
                        t.used = 0;
                    } else {
                        err = kErrPool;
                    }
                }
            } else {
                t.root = -1;
                t.used = 0;
            }
            if (kSession && !err && t.root >= 0 && static_cast<unsigned long long>(t.used) + minibatch_words(p) > p.pool_words) {
                t.root = -1;
                t.used = 0;
            }
        }
        if (!err && t.root < 0) {
            t.root = add_node(R, p, t, position);
            if (t.root < 0) err = kErrPool;
        }
        uint32_t noise_n = cmd.noise_n;
        if (!err) {
            float* nz = p.noise + static_cast<size_t>(si) * p.max_children;
            for (uint32_t i = static_cast<uint32_t>(ln); i < noise_n && i < p.max_children; i += DS_LANES) nz[i] = cmd_noise[i];
            wsync();
            const Hdr* rh = T::hdr(t.pool, t.root);
            if (reused && rh->expanded && rh->count > 0 && noise_n) {  // mod.rs:329-332
                if (noise_n == static_cast<uint32_t>(rh->count))
                    apply_noise(t.pool, t.root, rh->count, nz, p.noise_eps[cur]);
                else
                    err = kErrNoise;
                noise_n = 0;
            }
        }
        uint32_t kept = 0;  // sessions: the root's visits before the search
        if (kSession && !err) {
            const Hdr* rh = T::hdr(t.pool, t.root);
            int part = 0;
            if (rh->expanded)
                for (int i = ln; i < rh->count; i += DS_LANES) part += T::child(t.pool, t.root)[i].n;
            kept = static_cast<uint32_t>(wsum(part));
        }
        if (ln == 0) {
            root[cur] = t.root;
            used[cur] = t.used;
            S.root[0] = root[0];
            S.root[1] = root[1];
            S.used[0] = used[0];
            S.used[1] = used[1];
            S.buf[0] = buf[0];
            S.buf[1] = buf[1];
            S.hist_len = hist_len;
            S.cur = cur;
            S.sims_left = p.sim_num[cur];
            S.noise_n = noise_n;
            S.leaf = -1;
            S.path_len = 0;
            if (kSession) {
                S.sims_left = p.session->nodes;
                S.row = kept;
                S.pad[0] = 0;
                S.pad[1] = 0;
            }
            if (err) {
                atomic_or_u32(p.error, err);
                S.error = err;
                S.phase = kIdle;
            } else {
                S.phase = kRun | ((wave + p.begin_lead) << 2);
            }
        }
    }
};

}  // namespace ds
