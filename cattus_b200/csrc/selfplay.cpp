// Self-play driver: the caller side of the evaluation path (include/cattus_b200_selfplay.h).
//
// Restates, in host C++, the reference's MctsPlayer (engine/src/mcts/mod.rs:105-454), the Hex / TicTacToe rules
// (engine/src/hex/core.rs:112-335, engine/src/ttt/core.rs:101-246; chess: chess_rules.hpp), NNetwork::evaluate's flip +
// ValueFuncCache (engine/src/net/mod.rs:74-87,158-182; engine/src/mcts/cache.rs:31-75), the self-play game loop
// (training/self-play/src/self_play.rs:94-276), the .traindata writers (self_play.rs:33-61, serialize/hex.rs:16-28,
// serialize/ttt.rs:17-22, serialize/chess.rs:18-57) and the player behind the UCI loop (engine/src/chess/uci.rs).  The
// oracles it is tested against are oracle/mcts.py and oracle/chess.py.
//
// B200-first arrangement: a worker thread advances `games_per_thread` games as state machines.  Each game runs its
// simulations strictly in the reference's order (select -> evaluate -> expand -> backpropagate, one leaf in flight per
// tree), but when a game needs the network it parks and the worker moves on to its next game; once every game of the
// worker is parked, all their leaves go to the evaluator as one batch.  Nothing is shared between workers except the
// evaluator and its position cache, so there is no cross-thread rendezvous on the leaf path at all.
//
// Third-party behaviour reproduced on purpose (see oracle/mcts.py for the derivation):
//   * petgraph `edges()` iterates newest-edge-first and `Iterator::max_by` keeps the last maximum, so ties in `select`
//     and in the temperature-0 move choice go to the child that was inserted FIRST;
//   * `remove_all_but_subtree` re-inserts edges in iteration order, which reverses every kept node's child order at
//     each tree reuse.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/types.h>

#include "../../include/cattus_b200_selfplay.h"
#include "dsearch_api.hpp"
#include "sp_common.hpp"

namespace sp {

// ------------------------------------------------------------------------------------------------ rules
// status(): 0 ongoing, 1 Player1 won, 2 Player2 won, 3 draw
struct PosKeyHash {
    size_t operator()(const PosKey& k) const {
        auto mix = [](uint64_t x) {
            x ^= x >> 33;
            x *= 0xff51afd7ed558ccdull;
            x ^= x >> 33;
            return x;
        };
        uint64_t h = mix(static_cast<uint64_t>(k.a)) ^ (mix(static_cast<uint64_t>(k.a >> 64) + 0x9E3779B97F4A7C15ull) * 3);
        h ^= mix(static_cast<uint64_t>(k.b) + 0x632BE59BD9B4E019ull) * 5 ^ (mix(static_cast<uint64_t>(k.b >> 64) + 0x1234567ull) * 7);
        return static_cast<size_t>(mix(h));
    }
};

// ------------------------------------------------------------------------------------------------ cache
// ValueFuncCache (mcts/cache.rs:31-75): position -> (per-move probabilities in legal_moves() order, value).  A hit
// returns exactly what was stored.  Laid out for many worker threads instead of one RwLock<HashMap>: a flat
// set-associative table (8 ways per bucket, probabilities stored inline, striped spin locks), first-in-first-out
// eviction WITHIN a bucket instead of over the whole table.  Capacity is max_size rounded up to whole buckets.
// Eviction order only changes which later lookups hit, never a result (the evaluator is batch invariant).
class Cache {
  public:
    Cache(size_t max_size, int moves_num) : stride_(static_cast<size_t>(moves_num) + 1) {
        n_buckets_ = 1;
        while (n_buckets_ * kWays < max_size) n_buckets_ <<= 1;
        meta_ = static_cast<Meta*>(zeroed_huge(n_buckets_ * sizeof(Meta)));
        keys_ = static_cast<PosKey*>(zeroed_huge(n_buckets_ * kWays * sizeof(PosKey)));
        vals_ = static_cast<float*>(zeroed_huge(n_buckets_ * kWays * stride_ * sizeof(float)));
        if (!meta_ || !keys_ || !vals_) throw SpError{CATTUS_B200_ENOMEM, "cannot allocate the position cache"};
        for (auto& l : locks_) l.clear();
    }
    ~Cache() {
        free_huge(meta_, n_buckets_ * sizeof(Meta));
        free_huge(keys_, n_buckets_ * kWays * sizeof(PosKey));
        free_huge(vals_, n_buckets_ * kWays * stride_ * sizeof(float));
    }
    Cache(const Cache&) = delete;
    Cache& operator=(const Cache&) = delete;

    // requests the bucket of `k` (tags, first keys) so that a find / insert a little later does not stall on memory
    void prefetch(const PosKey& k) const {
        const size_t b = PosKeyHash()(k) & (n_buckets_ - 1);
        __builtin_prefetch(&meta_[b]);
        __builtin_prefetch(&keys_[b * kWays]);
        __builtin_prefetch(&keys_[b * kWays + 4]);
    }
    // copies the stored (probs..., value) of `k` into out[0 .. n_legal] and returns true on a hit
    bool find(const PosKey& k, int n_legal, float* out) {
        const uint64_t h = PosKeyHash()(k);
        const size_t b = h & (n_buckets_ - 1);
        const uint16_t tag = tag_of(h);
        Guard g(locks_[b & (kLocks - 1)]);
        const Meta& m = meta_[b];
        for (size_t w = 0; w < kWays; ++w)
            if (m.tag[w] == tag && keys_[b * kWays + w] == k) {
                std::memcpy(out, vals_ + (b * kWays + w) * stride_, sizeof(float) * (n_legal + 1));
                return true;
            }
        return false;
    }
    // stores val[0 .. n_legal] unless the key is already there (another thread got there first), in which case the
    // cached entry is copied back into `val` (cache.rs:52-63).  Returns true if it was inserted.
    bool insert(const PosKey& k, int n_legal, float* val) {
        const uint64_t h = PosKeyHash()(k);
        const size_t b = h & (n_buckets_ - 1);
        const uint16_t tag = tag_of(h);
        Guard g(locks_[b & (kLocks - 1)]);
        Meta& m = meta_[b];
        for (size_t w = 0; w < kWays; ++w)
            if (m.tag[w] == tag && keys_[b * kWays + w] == k) {
                std::memcpy(val, vals_ + (b * kWays + w) * stride_, sizeof(float) * (n_legal + 1));
                return false;
            }
        size_t victim = kWays;
        for (size_t w = 0; w < kWays; ++w)
            if (m.tag[w] == 0) {
                victim = w;
                break;
            }
        if (victim == kWays) {  // bucket full: first in, first out within the bucket
            victim = m.next;
            m.next = static_cast<uint16_t>((m.next + 1) % kWays);
        }
        m.tag[victim] = tag;
        keys_[b * kWays + victim] = k;
        std::memcpy(vals_ + (b * kWays + victim) * stride_, val, sizeof(float) * (n_legal + 1));
        return true;
    }

  private:
    // Zero pages straight from the kernel, backed by transparent huge pages where the system allows it (the table is
    // probed at random: with 4 KB pages nearly every probe is also a TLB miss).
    static void* zeroed_huge(size_t bytes) {
        const size_t len = (bytes + (2u << 20) - 1) & ~static_cast<size_t>((2u << 20) - 1);
        void* p = ::mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
        if (p == MAP_FAILED) return nullptr;
#ifdef MADV_HUGEPAGE
        ::madvise(p, len, MADV_HUGEPAGE);
#endif
        return p;
    }
    static void free_huge(void* p, size_t bytes) {
        if (p) ::munmap(p, (bytes + (2u << 20) - 1) & ~static_cast<size_t>((2u << 20) - 1));
    }
    static constexpr size_t kWays = 8, kLocks = 4096;
    // one 32-byte record per bucket: 16-bit tags (0 = empty way) filter the key compares, so a miss touches one line
    struct alignas(32) Meta {
        uint16_t tag[kWays];
        uint16_t next;  // FIFO cursor once the bucket is full (ways fill in order 0..7 first)
        uint16_t pad[7];
    };
    static uint16_t tag_of(uint64_t h) {
        const uint16_t t = static_cast<uint16_t>(h >> 48);
        return t ? t : 1;
    }
    struct Guard {
        std::atomic_flag& f;
        explicit Guard(std::atomic_flag& fl) : f(fl) {
            while (f.test_and_set(std::memory_order_acquire)) {
#if defined(__x86_64__)
                __builtin_ia32_pause();
#endif
            }
        }
        ~Guard() { f.clear(std::memory_order_release); }
    };
    size_t stride_, n_buckets_;
    Meta* meta_ = nullptr;
    PosKey* keys_ = nullptr;
    float* vals_ = nullptr;
    std::atomic_flag locks_[kLocks];
};

// One evaluator = the reference's NNetwork: a network behind a callback plus its own cache.
struct Evaluator {
    cattus_b200_eval_fn fn = nullptr;
    void* ctx = nullptr;
    cattus_b200_t* leaf_handle = nullptr;  // non-null: single-position requests use the per-leaf pinned queue
    cattus_b200_t* async_handle = nullptr; // non-null: batches go out with eval_batch_submit / _wait (kept in flight)
    uint32_t max_rows = 0xFFFFFFFFu;       // the handle's max_batch: speculative rows never grow a batch beyond one device batch
    std::unique_ptr<Cache> cache;
};

// ------------------------------------------------------------------------------------------------ tree
// select's inner step (mod.rs:211-226) for one node, structure-of-arrays so the compiler can vectorise it (two IEEE
// divisions per child dominate a simulation otherwise).  Per lane exactly the scalar operations of
// calc_selection_heuristic (mod.rs:233-244) in the reference's order: exploit = n == 0 ? 0 : w / n;
// explore = (ef * init) * (sqrt(parent_simcount) / (1 + n)).  Returns the child the reference picks: petgraph's
// edges() runs newest-first and max_by keeps the LAST maximum, i.e. the maximal child with the smallest insertion index.
__attribute__((target_clones("avx2", "default"))) static int select_child(const float* __restrict__ init, const float* __restrict__ w,
                                                                          const int32_t* __restrict__ n, int count, float ef,
                                                                          float* __restrict__ val) {
    int32_t simcount = 1;  // counts stay far below 2^31; signed so that the int -> float conversion is one instruction
    for (int i = 0; i < count; ++i) simcount += n[i];
    const float sq = std::sqrt(static_cast<float>(simcount));
    for (int i = 0; i < count; ++i) {
        const float nf = static_cast<float>(n[i]);
        const float exploit = n[i] == 0 ? 0.0f : w[i] / nf;
        const float explore = ef * init[i] * (sq / static_cast<float>(1 + n[i]));
        val[i] = exploit + explore;
    }
    float best = val[0];
    for (int i = 1; i < count; ++i) best = val[i] > best ? val[i] : best;
    for (int i = 0; i < count; ++i)
        if (val[i] == best) return i;
    return count - 1;  // only reachable with NaNs, which the reference asserts away (mod.rs:444)
}
// Search tree storage.  Every visited node is ONE 16-byte-aligned block of 32-bit words in `pool`:
//   Header { position, count, expanded } | init_score[count] (f32) | score_w[count] (f32) | simulations_n[count] (i32) |
//   edge[count] | move16[count] (chess only: 16-bit moves, two per word)
// with count = number of legal moves (known from the position when the node is first visited; the rows are filled in
// when its evaluation arrives) and edge = (child block offset / 4 + 1) in the low 24 bits (0: child not visited yet, its
// position is derived on demand) + the move in the high 8 (MctsNode / MctsEdge, mod.rs:21-56).  A node visit during
// select touches one run of cache lines, and the run can be requested as soon as the parent has picked the child.
template <class Pos, bool Wide = false>
struct Tree {
    struct alignas(16) Header {
        Pos pos;
        int32_t count;     // children (legal moves of pos; 0 for finished positions)
        int32_t expanded;  // rows are valid: create_children has run (mod.rs:246-262)
    };
    static constexpr int32_t kHdrWords = static_cast<int32_t>((sizeof(Header) + 15) / 16 * 4);
    std::vector<uint32_t> pool;
    int32_t root = -1;
    void clear() {
        pool.clear();
        root = -1;
    }
    Header& hdr(int32_t b) { return *reinterpret_cast<Header*>(pool.data() + b); }
    const Header& hdr(int32_t b) const { return *reinterpret_cast<const Header*>(pool.data() + b); }
    float* init_score(int32_t b) { return reinterpret_cast<float*>(pool.data() + b + kHdrWords); }
    float* score_w(int32_t b) { return init_score(b) + hdr(b).count; }
    int32_t* simulations_n(int32_t b) { return reinterpret_cast<int32_t*>(pool.data() + b + kHdrWords + 2 * hdr(b).count); }
    uint32_t* edge(int32_t b) { return pool.data() + b + kHdrWords + 3 * hdr(b).count; }
    uint16_t* move16(int32_t b) { return reinterpret_cast<uint16_t*>(pool.data() + b + kHdrWords + 4 * hdr(b).count); }
    static size_t block_words(int32_t count) {
        const size_t c = static_cast<size_t>(count);
        return kHdrWords + 4 * c + (Wide ? (c + 1) / 2 : 0);
    }
    static uint32_t pack_edge(int32_t child_block, uint8_t m) {
        return (child_block < 0 ? 0u : (static_cast<uint32_t>(child_block >> 2) + 1u)) | (static_cast<uint32_t>(m) << 24);
    }
    static int32_t edge_child(uint32_t e) { return (e & 0xFFFFFFu) ? static_cast<int32_t>(((e & 0xFFFFFFu) - 1u) << 2) : -1; }
    static uint8_t edge_move(uint32_t e) { return static_cast<uint8_t>(e >> 24); }
    // appends the block of a newly visited node (rows zeroed, not expanded) and returns its offset; invalidates pointers
    int32_t new_block(const Pos& pos, int32_t count) {
        const size_t b = pool.size();
        const size_t words = (block_words(count) + 3) & ~static_cast<size_t>(3);  // blocks stay 16-byte aligned
        if (b + words >= (static_cast<size_t>(0xFFFFFE) << 2)) throw SpError{CATTUS_B200_ERANGE, "search tree exceeds its 2^26-word address space"};
        pool.resize(b + words);
        Header& h = hdr(static_cast<int32_t>(b));
        h.pos = pos;
        h.count = count;
        h.expanded = 0;
        return static_cast<int32_t>(b);
    }
};

template <class Rules>
class Worker {
    using Pos = typename Rules::Pos;
    using Move = typename Rules::Move;
    using TreeT = Tree<Pos, Rules::kChess>;
    static constexpr bool kChess = Rules::kChess;

    struct SimCand {
        int32_t node, child;
        int rank;  // 0: the node's best unvisited alternative, 1: its second best, ...
    };
    struct Player {
        TreeT tree;
        // speculation (cfg.speculate): (node block, child index) candidates of this tree -- the best-prior children of the nodes
        // it expanded; consumed from spec_head
        std::vector<std::pair<int32_t, int32_t>> spec_queue;
        size_t spec_head = 0;
    };
    enum Phase { kIdle, kStartMove, kSimulate, kWaitEval };
    struct Slot {
        Phase phase = kIdle;
        uint32_t game_idx = 0;
        SplitMix64 rng;
        std::vector<Pos> history;
        Player players[2];
        int cur = 0;  // index into players of the side searching now
        uint32_t sims_left = 0;
        struct PathStep {
            int32_t w_idx;  // word index of the taken child's score_w in the tree's pool
            int32_t count;  // children of that node: simulations_n is `count` words further
            int32_t child;  // block of the node the step leads to
        };
        std::vector<PathStep> path;  // root -> leaf
        int32_t leaf = -1;
        bool leaf_flipped = false;
        Pos leaf_eval_pos;  // the position as sent to the network (Player1 to move)
        uint32_t wait_row = 0;  // row of the pending batch this slot is parked on
        int32_t sel_node = -1;  // block of the node the in-progress select stands on (-1: no simulation in progress)
        PosKey leaf_key{0, 0};        // cache key of the leaf being evaluated
        int32_t prepared_leaf = -1;   // block whose evaluation inputs (leaf_*) were set up early, at its first visit
        int leaf_n_legal = 0;
        uint32_t group = 0;     // slot group (one batch per group and evaluator)
        Clock::time_point search_t0;
        GameRecord rec;
        std::vector<std::pair<Pos, std::vector<std::pair<Move, float>>>> pending_entries;
        bool repetition = false;  // ChessGame::repetition_detected (chess/core.rs:441-449)
        std::vector<SimCand> sim_cands;  // speculation: candidates seen along the simulation in progress
    };
    struct Pending {  // one batch under construction for one evaluator
        std::vector<uint64_t> planes;
        std::vector<PosKey> keys;
        std::vector<uint8_t> n_legal;
        std::vector<uint8_t> legal;    // chess: one 235-byte legal-move bitmap per row
        std::vector<uint32_t> parked;  // slots waiting on this batch (each remembers its row)
        std::vector<uint32_t> table;   // open addressing: row + 1 of a key already in the batch (in-batch dedupe)
        std::vector<uint32_t> used;
        void init(size_t slots) {
            size_t cap = 16;
            while (cap < 4 * slots) cap <<= 1;
            table.assign(cap, 0);
        }
        // row of `k` in this batch, or -1 after reserving the table cell for the row about to be appended
        int32_t find_or_reserve(const PosKey& k) {
            const size_t mask = table.size() - 1;
            size_t h = PosKeyHash()(k) & mask;
            while (table[h]) {
                if (keys[table[h] - 1] == k) return static_cast<int32_t>(table[h] - 1);
                h = (h + 1) & mask;
            }
            table[h] = static_cast<uint32_t>(keys.size()) + 1;
            used.push_back(static_cast<uint32_t>(h));
            return -1;
        }
        void clear() {
            planes.clear();
            keys.clear();
            n_legal.clear();
            legal.clear();
            parked.clear();
            for (uint32_t h : used) table[h] = 0;
            used.clear();
        }
    };
    // Slots can be split into groups (cfg.groups_per_thread); each group owns one batch under construction per evaluator
    // and may have one batch in flight per evaluator, so that while a group's leaves are on the GPU the worker simulates
    // the next group.  Small groups keep a worker's trees in cache (per-thread simulation rate 1.15 M/s with 256 games
    // in one group vs 1.6-1.7 M/s with 16-32, measured with 4 threads), but every batch costs ~20 us of CUDA calls, and
    // with all cores busy the two effects cancel: the default stays one group.
    struct Group {
        uint32_t first = 0, count = 0;
        Pending pend[2];
        int32_t ticket[2] = {-1, -1};
        uint32_t inflight_n[2] = {0, 0};
    };
    struct Counters {
        uint64_t simulations = 0, searches = 0, evaluations = 0, cache_hits = 0, cache_misses = 0, batches = 0, terminal = 0, speculative = 0;
        uint32_t w1 = 0, w2 = 0, d = 0, games = 0;
    };

  public:
    Worker(const Rules& rules, const cattus_b200_selfplay_cfg& cfg, const Params params[2], Evaluator* evals[2], Shared& sh)
        : R(rules), cfg_(cfg), sh_(sh) {
        params_[0] = params[0];
        params_[1] = params[1];
        evals_[0] = evals[0];
        evals_[1] = evals[1];
        // no more concurrent games per worker than an even split of this call's games (else the first workers take them all)
        const uint32_t stride = std::max<uint32_t>(1, cfg.game_stride), threads = std::max<uint32_t>(1, cfg.threads);
        const uint32_t my_games = cfg.games_num > cfg.first_game ? (cfg.games_num - cfg.first_game + stride - 1) / stride : 0;
        slots_.resize(std::max<uint32_t>(1, std::min<uint32_t>(cfg.games_per_thread, (my_games + threads - 1) / threads)));
        const bool async = evals[0]->async_handle != nullptr && (evals[1] == evals[0] || evals[1]->async_handle != nullptr);
        // measured (16 threads, hex5): 1 group x 256 games 13.2 M sims/s, 2 x 128 13.2 M, 4 x 64 11.3 M, 8 x 32 6.6 M --
        // the per-batch submission cost outweighs the better cache locality of small groups, so the default is one group
        uint32_t n_groups = cfg.groups_per_thread ? cfg.groups_per_thread : 1;
        n_groups = std::max<uint32_t>(1, std::min<uint32_t>({n_groups, static_cast<uint32_t>(slots_.size()), async ? 64u : 1u}));
        groups_.resize(n_groups);
        const uint32_t per = (static_cast<uint32_t>(slots_.size()) + n_groups - 1) / n_groups;
        for (uint32_t g = 0; g < n_groups; ++g) {
            Group& gr = groups_[g];
            gr.first = std::min<uint32_t>(g * per, static_cast<uint32_t>(slots_.size()));
            gr.count = std::min<uint32_t>(per, static_cast<uint32_t>(slots_.size()) - gr.first);
            gr.pend[0].init(gr.count);
            gr.pend[1].init(gr.count);
            for (uint32_t i = 0; i < gr.count; ++i) slots_[gr.first + i].group = g;
        }
        if (cfg.speculate) set_speculation(cfg.speculate);
        val_.resize(static_cast<size_t>(R.max_children()) + 1);
        if (const char* e = std::getenv("CATTUS_B200_SELFPLAY_RING")) ring_size_ = std::max(1, std::min<int>(kMaxRing, std::atoi(e)));
        abi_wpp_ = (R.moves_num() + 63) / 64;
    }

    void run() {
        try {
            for (auto& s : slots_) start_next_game(s);
            for (;;) {
                bool any = false, outstanding = false;
                for (Group& gr : groups_) {
                    for (int e = 0; e < 2; ++e)
                        if (gr.ticket[e] >= 0) collect(gr, e);
                    any |= run_group(gr);
                    if (sh_.failed.load(std::memory_order_relaxed)) {
                        drain_all();
                        return;
                    }
                    if (speculate_) fill_small_batches(gr);
                    for (int e = 0; e < 2; ++e)
                        if (!gr.pend[e].keys.empty()) {
                            send(gr, e);
                            outstanding = true;
                        }
                }
                if (!any && !outstanding) break;
            }
        } catch (const SpError& e) {
            fail(e.code, e.msg);
        } catch (const std::bad_alloc&) {
            fail(CATTUS_B200_ENOMEM, "out of host memory in a self-play worker (search trees / batch rows)");
        } catch (const std::exception& e) {
            fail(CATTUS_B200_EINVAL, std::string("self-play worker: ") + e.what());
        } catch (...) {
            fail(CATTUS_B200_EINVAL, "self-play worker: unknown exception");
        }
        std::lock_guard<std::mutex> g(sh_.mu);
        sh_.eval_wait += eval_wait_;
        sh_.simulations += c_.simulations;
        sh_.searches += c_.searches;
        sh_.evaluations += c_.evaluations;
        sh_.cache_hits += c_.cache_hits;
        sh_.cache_misses += c_.cache_misses;
        sh_.batches += c_.batches;
        sh_.terminal += c_.terminal;
        sh_.speculative += c_.speculative;
        sh_.w1 += c_.w1;
        sh_.w2 += c_.w2;
        sh_.d += c_.d;
        sh_.games += c_.games;
    }

    // One search at a time on slot 0, driven from outside: GamePlayer::next_move(pos_history) as the reference's UCI loop
    // calls it per `go` (engine/src/chess/uci.rs:158-161, mcts/mod.rs:448-454).  The tree is kept between calls and reused
    // when the new position is found in it (mod.rs:335-352).  Returns false if the position has no move to search.
    struct SearchStats {
        uint64_t simulations = 0, evaluations = 0, cache_hits = 0, terminal = 0;
        double seconds = 0.0;
        uint32_t root_visits_best = 0, root_children = 0, speculative = 0;
    };
    // Search sessions only: while a leaf waits for the network, up to `rows` more positions ride in the same evaluator call
    // and land in the cache -- the best-prior unvisited children of recently expanded nodes, which is where the next visits
    // of those nodes go (all their children have n = 0, so select picks the largest prior).  The cache returns exactly what
    // a fresh evaluation returns (the evaluator is batch invariant), so the search is unchanged; only its waiting is.
    void set_speculation(uint32_t rows) {
        speculate_ = std::min<uint32_t>(rows, 255);
        for (Group& gr : groups_)  // the in-batch dedupe tables must hold the extra rows too
            for (Pending& pb : gr.pend) pb.init(gr.count + std::max<uint32_t>(speculate_, kSpecTargetRows));
    }
    void reseed(uint64_t seed) { slots_[0].rng = SplitMix64(game_seed(seed, 0)); }
    bool search_from(const std::vector<Pos>& history, Move* best, SearchStats* stats) {
        Slot& s = slots_[0];
        // a previous `go` may have ended in an evaluator error mid-search: nothing of it may survive into this one (a stale
        // pending row would be delivered twice and the simulation counter would wrap)
        drain_all();
        for (Group& g : groups_)
            for (Pending& pb : g.pend) pb.clear();
        s.phase = kIdle;
        s.sel_node = -1;
        s.path.clear();
        s.sim_cands.clear();
        s.prepared_leaf = -1;
        s.history = history;
        s.pending_entries.clear();
        s.rec.moves.clear();
        s.repetition = false;
        if (R.status(s.history.back()) != 0) return false;
        const Counters before = c_;
        const auto t0 = Clock::now();
        s.cur = 0;
        begin_search(s);
        s.phase = kSimulate;
        s.sel_node = -1;
        const uint64_t spec_before = c_.speculative;
        Group& gr = groups_[0];
        while (s.phase != kStartMove) {
            if (!step(0)) {  // parked on the evaluator: evaluate now (one leaf in flight, like the reference)
                add_speculative_rows(s, gr, std::min(speculate_, evals_[0]->max_rows - 1));
                for (int e = 0; e < 2; ++e)
                    if (!gr.pend[e].keys.empty()) send(gr, e);
            }
        }
        if (sh_.failed.load()) return false;
        *best = static_cast<Move>(s.rec.moves.back());
        if (stats) {
            stats->simulations = c_.simulations - before.simulations;
            stats->evaluations = c_.evaluations - before.evaluations;
            stats->cache_hits = c_.cache_hits - before.cache_hits;
            stats->terminal = c_.terminal - before.terminal;
            stats->seconds = std::chrono::duration<double>(Clock::now() - t0).count();
            const auto& probs = s.pending_entries.back().second;
            stats->root_children = static_cast<uint32_t>(probs.size());
            float top = 0.0f;
            for (auto& mp : probs) top = std::max(top, mp.second);
            stats->root_visits_best = static_cast<uint32_t>(top * static_cast<float>(params_[0].sim_num) + 0.5f);
            stats->speculative = static_cast<uint32_t>(c_.speculative - spec_before);
        }
        return true;
    }

  private:
    // error path of run(): every ticket in flight is waited, the first error of the job is kept, the other workers stop
    void fail(int code, const std::string& msg) noexcept {
        try {
            drain_all();
        } catch (...) {
        }
        std::lock_guard<std::mutex> g(sh_.mu);
        if (!sh_.failed.exchange(true)) {
            sh_.error_code = code;
            sh_.error = msg;
        }
    }

    // ---------------------------------------------------------------- game loop (self_play.rs:179-246)
    void start_next_game(Slot& s) {
        const uint32_t stride = std::max<uint32_t>(1, cfg_.game_stride);
        const uint32_t k = sh_.next_game.fetch_add(1);
        const uint64_t idx = static_cast<uint64_t>(cfg_.first_game) + static_cast<uint64_t>(k) * stride;
        if (idx >= cfg_.games_num) {
            s.phase = kIdle;
            return;
        }
        s.game_idx = static_cast<uint32_t>(idx);
        s.rng = SplitMix64(game_seed(cfg_.seed, s.game_idx));
        s.history.clear();
        s.history.push_back(R.initial());
        s.players[0].tree.clear();
        s.players[1].tree.clear();
        s.rec = GameRecord();
        s.rec.game_idx = s.game_idx;
        s.pending_entries.clear();
        s.repetition = false;
        s.phase = kStartMove;
    }

    // The games of a group are advanced INTERLEAVED: a ring of `ring_size_` games each does one small step per turn (one level
    // of select, split into "request the node's child rows" and "pick the child"), so that the cache misses of one
    // game's tree walk overlap with the work of the others -- with hundreds of trees per worker nearly every node
    // visit is a miss.  Each game still runs its own simulations strictly in order; only the interleaving between
    // games changes, which no result depends on.
    bool run_group(Group& gr) {
        bool any = false;
        uint32_t ring[kMaxRing];
        uint32_t in_ring = 0, next = 0;
        auto admit = [&]() {
            while (next < gr.count && in_ring < ring_size_) {
                const uint32_t i = gr.first + next++;
                const Slot& s = slots_[i];
                if (s.phase == kIdle) continue;
                any = true;
                if (s.phase == kWaitEval) continue;
                ring[in_ring++] = i;
            }
        };
        admit();
        while (in_ring) {
            for (uint32_t r = 0; r < in_ring;) {
                if (step(ring[r])) {
                    ++r;
                } else {  // parked on the evaluator or out of games: hand the ring place to the next game of the group
                    ring[r] = ring[--in_ring];
                    admit();
                }
            }
        }
        return any;
    }

    // One small unit of work for game `si`; false when the game left the runnable state (parked or idle).
    bool step(uint32_t si) {
        Slot& s = slots_[si];
        if (s.phase == kStartMove) {
            const Pos& pos = s.history.back();
            int st = s.repetition ? 3 : R.status(pos);  // ChessGame::status: a threefold repetition is a draw
            if (st == 0 && cfg_.max_moves && s.rec.moves.size() >= cfg_.max_moves) st = 3;  // bounded runs only (not in the reference)
            if (st != 0) {
                finish_game(s, st);
                start_next_game(s);
                return s.phase != kIdle;
            }
            int who = pos.turn;  // self_play.rs:198-205
            if (s.game_idx % 2 == 1) who = 3 - who;
            s.cur = who - 1;
            begin_search(s);
            s.phase = kSimulate;
            s.sel_node = -1;
            return true;
        }
        // kSimulate
        TreeT& t = s.players[s.cur].tree;
        if (s.sel_node < 0) {
            if (s.sims_left == 0) {
                end_search(s);
                s.phase = kStartMove;
                return true;
            }
            s.path.clear();  // select (mod.rs:199-231) starts at the root
            s.sim_cands.clear();
            s.prepared_leaf = -1;
            s.sel_node = t.root;
            prefetch_block(t, t.root, t.hdr(t.root).count);
            // a first visit appends a block at the tail of the pool: request those lines for writing
            if (t.pool.capacity() >= t.pool.size() + 128)
                for (int off = 0; off < 128; off += 16) __builtin_prefetch(t.pool.data() + t.pool.size() + off, 1);
            return true;
        }
        const int32_t node = s.sel_node;
        const typename TreeT::Header& nd = t.hdr(node);
        if (!nd.expanded || R.status(nd.pos) != 0) {
            s.sel_node = -1;
            if (at_leaf(s, node)) return true;  // terminal: backpropagated
            return evaluate_leaf(si);
        }
        const int32_t count = nd.count;
        const int32_t best = select_child(t.init_score(node), t.score_w(node), t.simulations_n(node), count, params_[s.cur].explore_factor, sel_);
        {
            if (speculate_) {  // the best-scoring children of this node that have no node yet, other than the one taken: likely next leaves
                const uint32_t* ed = t.edge(node);
                int32_t alt[kSpecPerLevel];
                int n_alt = 0;
                for (int32_t i = 0; i < count; ++i) {
                    if (i == best || TreeT::edge_child(ed[i]) >= 0) continue;
                    int at = n_alt;  // insertion into the short list sorted by descending score
                    while (at > 0 && sel_[i] > sel_[alt[at - 1]]) --at;
                    if (at >= kSpecPerLevel) continue;
                    for (int k = std::min(n_alt, kSpecPerLevel - 1); k > at; --k) alt[k] = alt[k - 1];
                    alt[at] = i;
                    n_alt = std::min(n_alt + 1, kSpecPerLevel);
                }
                for (int k = 0; k < n_alt; ++k) s.sim_cands.push_back({node, alt[k], k});
            }
        }
        int32_t c = TreeT::edge_child(t.edge(node)[best]);
        if (c < 0) {
            c = materialise(t, node, best);
            prepare_leaf(s, t, c);  // a first visit is this simulation's leaf: set up its evaluation and request its cache bucket now
        } else {
            prefetch_block(t, c, count);
        }
        s.path.push_back({node + TreeT::kHdrWords + count + best, count, c});
        s.sel_node = c;
        return true;
    }

    // requests a node's header and the three arrays select reads; `children` is the caller's estimate of the node's
    // child count (its parent's: each move removes one legal move in hex and tic-tac-toe)
    static void prefetch_block(const TreeT& t, int32_t b, int32_t children) {
        const uint32_t* p = t.pool.data() + b;
        const int words = TreeT::kHdrWords + 3 * children;
        for (int off = 0; off < words; off += 16) __builtin_prefetch(p + off);
    }

    void finish_game(Slot& s, int status) {
        const uint8_t winner = status == 3 ? 0 : static_cast<uint8_t>(status);
        s.rec.winner = winner;
        for (size_t pos_idx = 0; pos_idx < s.pending_entries.size(); ++pos_idx) {
            auto& pe = s.pending_entries[pos_idx];
            std::vector<uint8_t> bytes;
            const int dir = make_entry(R, s.game_idx, pe.first, pe.second, winner, bytes);
            if (cfg_.out_dir1 && cfg_.out_dir2) write_entry_file(dir == 1 ? cfg_.out_dir1 : cfg_.out_dir2, s.game_idx, pos_idx, bytes);
            if (cfg_.keep_records) {
                s.rec.entries.push_back(std::move(bytes));
                s.rec.entry_dir.push_back(static_cast<uint8_t>(dir));
            }
        }
        // winner counters: self_play.rs:226-241
        uint8_t credited = winner;
        if (credited && s.game_idx % 2 == 1) credited = static_cast<uint8_t>(3 - credited);
        if (credited == 0)
            c_.d += 1;
        else if (credited == 1)
            c_.w1 += 1;
        else
            c_.w2 += 1;
        c_.games += 1;
        if (cfg_.keep_records) {
            std::lock_guard<std::mutex> g(sh_.mu);
            sh_.records.push_back(std::move(s.rec));
        }
    }

    // ---------------------------------------------------------------- MctsPlayer
    // calc_moves_probabilities up to develop_tree (mod.rs:335-362)
    void begin_search(Slot& s) {
        s.search_t0 = Clock::now();
        TreeT& t = s.players[s.cur].tree;
        const Pos& position = s.history.back();
        if (t.root >= 0) {
            const int32_t node = find_node_with_position(t, position);
            if (node >= 0)
                remove_all_but_subtree(s, t, node);
            else
                t.clear();
        }
        if (t.root < 0) {
            t.pool.reserve((static_cast<size_t>(params_[s.cur].sim_num) + 8) * TreeT::block_words(typical_children()));
            t.root = add_node(t, position);
        }
        s.sims_left = params_[s.cur].sim_num;
        s.players[s.cur].spec_queue.clear();  // block offsets of the tree before reuse
        s.players[s.cur].spec_head = 0;
    }

    // mod.rs:283-301, depth_limit = 3 (root, its children, their children).  Unvisited children have no node yet;
    // their position is parent + move, compared on the fly and materialised on a match.
    int32_t find_node_with_position(TreeT& t, const Pos& position) {
        if (R.same(t.hdr(t.root).pos, position)) return t.root;
        std::vector<int32_t> layer{t.root}, next;
        for (int depth = 1; depth < 3; ++depth) {
            next.clear();
            for (int32_t n : layer) {
                if (!t.hdr(n).expanded) continue;
                const int32_t count = t.hdr(n).count;
                for (int32_t i = count - 1; i >= 0; --i) {
                    const uint32_t e = t.edge(n)[i];
                    const int32_t c = TreeT::edge_child(e);
                    if (c >= 0) {
                        if (R.same(t.hdr(c).pos, position)) return c;
                        next.push_back(c);
                    } else if (child_matches(t.hdr(n).pos, move_at(t, n, i), position)) {
                        return materialise(t, n, i);
                    }
                }
            }
            layer.swap(next);
        }
        return -1;
    }

    // block size hint: every hex / tic-tac-toe node could have all cells free; a chess position has ~35 moves
    int32_t typical_children() const { return kChess ? 48 : R.moves_num(); }

    Move move_at(TreeT& t, int32_t node, int32_t i) const {
        if constexpr (kChess)
            return t.move16(node)[i];
        else
            return TreeT::edge_move(t.edge(node)[i]);
    }
    bool child_matches(const Pos& parent, Move m, const Pos& target) const {
        if constexpr (kChess)
            return Rules::same(R.moved(parent, m), target);
        else
            return R.child_matches(parent, m, target);
    }

    // Appends the block of a node visited for the first time.  Its child count is the number of legal moves (0 for a
    // finished position); for chess the moves themselves are generated here, once, in the order NNetwork::evaluate
    // returns them, and kept in the block.
    int32_t add_node(TreeT& t, const Pos& pos) {
        if constexpr (kChess) {
            Pos p = pos;
            Move buf[256];
            const int32_t n = R.children(p, buf);
            const int32_t b = t.new_block(p, n);
            if (n) std::memcpy(t.move16(b), buf, sizeof(Move) * n);
            return b;
        } else {
            return t.new_block(pos, R.status(pos) != 0 ? 0 : popcount128(R.legal_mask(pos)));
        }
    }

    int32_t materialise(TreeT& t, int32_t parent, int32_t i) {
        const Move m = move_at(t, parent, i);
        const Pos child = R.moved(t.hdr(parent).pos, m);
        const int32_t cb = add_node(t, child);
        t.edge(parent)[i] = TreeT::pack_edge(cb, kChess ? 0 : static_cast<uint8_t>(m));
        return cb;
    }

    // mod.rs:303-333: copy the subtree; edges are re-inserted in iteration (newest-first) order => reversed
    void remove_all_but_subtree(Slot& s, TreeT& t, int32_t sub_root) {
        if (t.root == sub_root) return;
        TreeT nt;
        // The copy goes into a recycled buffer (every move of every game replaces a tree: fresh allocations of ~1 MB
        // each mean an mmap, a few hundred page faults and an munmap per move); room for the kept subtree plus one
        // more search.
        if (!pool_free_.empty()) {
            nt.pool = std::move(pool_free_.back());
            pool_free_.pop_back();
            nt.pool.clear();
        }
        nt.pool.reserve(t.pool.size() / 4 + (static_cast<size_t>(params_[s.cur].sim_num) + 8) * TreeT::block_words(typical_children()));
        nt.root = nt.new_block(t.hdr(sub_root).pos, t.hdr(sub_root).count);
        std::vector<std::pair<int32_t, int32_t>> stack{{sub_root, nt.root}};
        while (!stack.empty()) {
            const auto [old_n, new_n] = stack.back();
            stack.pop_back();
            if (!t.hdr(old_n).expanded) {
                // visited but never expanded: no edges yet, so nothing to reverse -- its moves keep their generated order
                if constexpr (kChess) std::memcpy(nt.move16(new_n), t.move16(old_n), sizeof(Move) * t.hdr(old_n).count);
                continue;
            }
            const int32_t count = t.hdr(old_n).count;
            nt.hdr(new_n).expanded = 1;
            for (int32_t i = 0; i < count; ++i) {  // new insertion order = old iteration order (newest first)
                const int32_t o = count - 1 - i;
                if constexpr (kChess) nt.move16(new_n)[i] = t.move16(old_n)[o];
                const uint32_t e = t.edge(old_n)[o];
                nt.init_score(new_n)[i] = t.init_score(old_n)[o];
                nt.score_w(new_n)[i] = t.score_w(old_n)[o];
                nt.simulations_n(new_n)[i] = t.simulations_n(old_n)[o];
                int32_t nc = -1;
                const int32_t old_c = TreeT::edge_child(e);
                if (old_c >= 0) {
                    nc = nt.new_block(t.hdr(old_c).pos, t.hdr(old_c).count);  // may move nt.pool: pointers are re-derived below
                    stack.push_back({old_c, nc});
                }
                nt.edge(new_n)[i] = TreeT::pack_edge(nc, TreeT::edge_move(e));
            }
        }
        pool_free_.push_back(std::move(t.pool));
        t = std::move(nt);
        if (t.hdr(t.root).expanded && t.hdr(t.root).count > 0) add_dirichlet_noise(s, t, t.root);
    }

    // mod.rs:419-446
    void add_dirichlet_noise(Slot& s, TreeT& t, int32_t node) {
        const Params& P = params_[s.cur];
        if (P.noise_alpha == 0.0f || P.noise_eps == 0.0f) return;
        const int32_t count = t.hdr(node).count;
        if (count < 2) return;
        const double tot = draw_noise(s.rng, P.noise_alpha, count, noise_);
        const float eps = P.noise_eps;
        for (int i = 0; i < count; ++i) {  // zip(edges() order = newest first, noise)
            float& init = t.init_score(node)[count - 1 - i];
            const float nz = static_cast<float>(noise_[i] / tot);
            init = (1.0f - eps) * init + eps * nz;
        }
    }

    // The rest of one develop_tree iteration once select has reached `node` (mod.rs:162-195), first half: terminal
    // leaves are backpropagated at once (returns true); otherwise the position to evaluate and its cache key are set up.
    bool at_leaf(Slot& s, int32_t node) {
        TreeT& t = s.players[s.cur].tree;
        s.leaf = node;
        if constexpr (kChess) {
            if (detect_repetition(s, t)) {  // mod.rs:162,174-175: scored as a draw, the leaf stays as it is
                c_.terminal += 1;
                backpropagate(s, t, 0.0f);
                return true;
            }
        }
        const Pos leaf_pos = t.hdr(node).pos;
        const int st = R.status(leaf_pos);
        if (st != 0) {
            c_.terminal += 1;
            backpropagate(s, t, st == 3 ? 0.0f : (st == 1 ? 1.0f : -1.0f));
            return true;
        }
        if (s.prepared_leaf != node) prepare_leaf(s, t, node);
        return false;
    }

    // MctsPlayer::detect_repetition (mod.rs:133-154): does any position occur REPETITION_LIMIT (3) times in the game's
    // history followed by the positions along the selected path?  The history alone never does (the game would be over),
    // so each path position is counted against what precedes it; equal positions lie an even number of plies apart and
    // not beyond the last pawn move or capture (`rev`).
    bool detect_repetition(const Slot& s, TreeT& t) const {
        const int32_t H = static_cast<int32_t>(s.history.size());
        for (int32_t j = 0; j < static_cast<int32_t>(s.path.size()); ++j) {
            const Pos& p = t.hdr(s.path[j].child).pos;
            int seen = 1;
            for (int32_t d = 2; d <= p.rev; d += 2) {
                const int32_t idx = H + j - d;
                if (idx < 0) break;
                const Pos& q = idx >= H ? t.hdr(s.path[idx - H].child).pos : s.history[idx];
                if (Rules::same(p, q) && ++seen >= 3) return true;
            }
        }
        return false;
    }

    // NNetwork::evaluate (net/mod.rs:74-87), first part: flip to the side-to-move view, cache key, legal count
    void prepare_leaf(Slot& s, TreeT& t, int32_t node) {
        const Pos& leaf_pos = t.hdr(node).pos;
        s.prepared_leaf = node;
        if (R.status(leaf_pos) != 0) return;
        s.leaf_flipped = leaf_pos.turn != 1;
        if constexpr (kChess) {
            uint64_t q[4];  // the stored position already is the evaluator's view
            R.key_planes(leaf_pos, q);
            s.leaf_key = PosKey{static_cast<u128>(q[0]) | (static_cast<u128>(q[1]) << 64), static_cast<u128>(q[2]) | (static_cast<u128>(q[3]) << 64)};
        } else {
            s.leaf_eval_pos = s.leaf_flipped ? R.flipped_boards(leaf_pos) : leaf_pos;
            s.leaf_key = R.key(s.leaf_eval_pos);
        }
        s.leaf_n_legal = t.hdr(node).count;
        if (evals_[s.cur]->cache) evals_[s.cur]->cache->prefetch(s.leaf_key);
    }

    // cache lookup, else join the group's batch.  Returns false if the leaf was parked on the evaluator.
    bool evaluate_leaf(uint32_t si) {
        Slot& s = slots_[si];
        Evaluator& ev = *evals_[s.cur];
        const PosKey key = s.leaf_key;
        const int n_legal = s.leaf_n_legal;
        if (ev.cache && ev.cache->find(key, n_legal, val_.data())) {
            c_.cache_hits += 1;
            deliver(s, val_.data());
            return true;
        }
        Pending& pb = groups_[s.group].pend[evals_[0] == evals_[1] ? 0 : s.cur];
        const int32_t row = pb.find_or_reserve(key);
        if (row >= 0) {
            s.wait_row = static_cast<uint32_t>(row);
            if (ev.cache) c_.cache_hits += 1;  // the reference would find it cached by the time it computed it
        } else {
            s.wait_row = static_cast<uint32_t>(pb.keys.size());
            pb.keys.push_back(key);
            if constexpr (kChess) {
                TreeT& t = s.players[s.cur].tree;
                uint64_t pl[Rules::kPlanes];
                R.planes(t.hdr(s.leaf).pos, pl);
                pb.planes.insert(pb.planes.end(), pl, pl + Rules::kPlanes);
                const size_t at = pb.legal.size();
                pb.legal.resize(at + Rules::kLegalBytes, 0);
                const Move* mv = t.move16(s.leaf);
                for (int k = 0; k < n_legal; ++k) {
                    const int idx = R.nn_idx(mv[k]);
                    pb.legal[at + (idx >> 3)] |= static_cast<uint8_t>(1u << (idx & 7));
                }
            } else {
                u128 pl[3];
                R.planes(s.leaf_eval_pos, pl);
                for (int c = 0; c < 3; ++c)
                    for (int k = 0; k < abi_wpp_; ++k) pb.planes.push_back(static_cast<uint64_t>(pl[c] >> (64 * k)));
            }
            pb.n_legal.push_back(static_cast<uint8_t>(n_legal));
        }
        pb.parked.push_back(si);
        s.phase = kWaitEval;
        return false;
    }

    // create_children + root noise + backpropagate for a leaf whose evaluation is known (mod.rs:180-194, :246-262)
    void deliver(Slot& s, const float* val) {
        TreeT& t = s.players[s.cur].tree;
        const int32_t leaf = s.leaf;
        const int32_t count = t.hdr(leaf).count;  // the legal moves: the block was sized when the node was first visited
        if constexpr (kChess) {
            // calc_moves_probs (net/mod.rs:106-119) gathers per legal move; the evaluator returns the probabilities compact in
            // ascending nn index, so child i takes the entry at the rank of its nn index among the legal ones
            const Move* mv = t.move16(leaf);
            constexpr int kWords = (Rules::kMovesNum + 63) / 64;
            uint64_t bits[kWords] = {0};
            uint16_t idx[256], before[kWords];
            for (int32_t i = 0; i < count; ++i) {
                idx[i] = static_cast<uint16_t>(R.nn_idx(mv[i]));
                bits[idx[i] >> 6] |= 1ull << (idx[i] & 63);
            }
            uint16_t run = 0;
            for (int w = 0; w < kWords; ++w) {
                before[w] = run;
                run = static_cast<uint16_t>(run + __builtin_popcountll(bits[w]));
            }
            float* init = t.init_score(leaf);
            for (int32_t i = 0; i < count; ++i)
                init[i] = val[before[idx[i] >> 6] + __builtin_popcountll(bits[idx[i] >> 6] & ((1ull << (idx[i] & 63)) - 1))];
        } else {
        const u128 legal = R.legal_mask(s.leaf_eval_pos);
        std::memcpy(t.init_score(leaf), val, sizeof(float) * count);
        uint32_t* ed = t.edge(leaf);
        int32_t k = 0;
        for (int half = 0; half < 2; ++half) {  // legal_moves() of the evaluated position, ascending; un-flipped by flip_score_if_needed
            uint64_t bits = static_cast<uint64_t>(legal >> (64 * half));
            while (bits) {
                const int m = 64 * half + __builtin_ctzll(bits);
                bits &= bits - 1;
                ed[k++] = TreeT::pack_edge(-1, static_cast<uint8_t>(s.leaf_flipped ? R.flip_move(m) : m));
            }
        }
        }
        t.hdr(leaf).expanded = 1;
        if (leaf == t.root) add_dirichlet_noise(s, t, leaf);
        {
            if (speculate_ && count > 0) {  // remember this node's two best-prior children as candidates to evaluate ahead
                const float* init = t.init_score(leaf);
                int32_t a = 0, b = -1;
                for (int32_t i = 1; i < count; ++i) {
                    if (init[i] > init[a]) {
                        b = a;
                        a = i;
                    } else if (b < 0 || init[i] > init[b]) {
                        b = i;
                    }
                }
                Player& pl = s.players[s.cur];
                pl.spec_queue.emplace_back(leaf, a);
                if (b >= 0) pl.spec_queue.emplace_back(leaf, b);
            }
        }
        float v = val[count];
        if (s.leaf_flipped) v = -v;
        backpropagate(s, t, v);
    }

    // mod.rs:270-281
    void backpropagate(Slot& s, TreeT& t, float score) {
        const uint8_t root_turn = t.hdr(t.root).pos.turn;  // the side to move alternates along the path in hex and tic-tac-toe
        for (size_t i = 0; i < s.path.size(); ++i) {
            const uint8_t turn = (i & 1) ? static_cast<uint8_t>(3 - root_turn) : root_turn;
            reinterpret_cast<int32_t*>(t.pool.data())[s.path[i].w_idx + s.path[i].count] += 1;
            reinterpret_cast<float*>(t.pool.data())[s.path[i].w_idx] += turn == 1 ? score : -score;
        }
        s.sims_left -= 1;
        c_.simulations += 1;
    }

    // the rest of calc_moves_probabilities + choose_move_from_probabilities + the game step (mod.rs:364-417,
    // self_play.rs:207-217)
    void end_search(Slot& s) {
        TreeT& t = s.players[s.cur].tree;
        const Params& P = params_[s.cur];
        const typename TreeT::Header& root = t.hdr(t.root);
        std::vector<std::pair<Move, float>> probs;
        probs.reserve(root.count);
        uint32_t total = 0;
        const int32_t* rn = t.simulations_n(t.root);
        for (int32_t i = 0; i < root.count; ++i) total += static_cast<uint32_t>(rn[i]);
        for (int32_t i = root.count - 1; i >= 0; --i)  // edges() order
            probs.emplace_back(move_at(t, t.root, i), static_cast<float>(rn[i]) / static_cast<float>(total));
        const double secs = std::chrono::duration<double>(Clock::now() - s.search_t0).count();
        {
            std::lock_guard<std::mutex> g(sh_.mu);  // RunningAverage(0.99), util/metric.rs:1-20
            sh_.search_duration = (1.0 - 0.99) * sh_.search_duration + 0.99 * secs;
        }
        c_.searches += 1;
        if (probs.empty()) throw SpError{CATTUS_B200_EINVAL, "search produced no moves"};
        const int chosen = choose_move(P, s.history.size(), probs, s.rng, weights_);  // choose_move_from_probabilities
        const Move mv = probs[chosen].first;
        s.pending_entries.emplace_back(s.history.back(), std::move(probs));
        if constexpr (kChess) {
            s.rec.moves.push_back(Rules::real_move(s.history.back(), mv));
            Pos np = R.moved(s.history.back(), mv);
            Move buf[256];
            R.children(np, buf);  // settles status()
            // ChessGame::play_single_turn (chess/core.rs:441-449): the third occurrence of a position ends the game
            int seen = 1;
            const int32_t H = static_cast<int32_t>(s.history.size());
            for (int32_t d = 2; d <= np.rev && d <= H; d += 2)
                if (Rules::same(np, s.history[H - d])) ++seen;
            if (seen >= 3) s.repetition = true;
            s.history.push_back(np);
        } else {
            s.rec.moves.push_back(mv);
            s.history.push_back(R.moved(s.history.back(), mv));
        }
    }

    // Speculation (cfg.speculate).  A device batch of 1 ... 256 positions costs the same time, so while leaves wait for the
    // network, positions that are likely to be asked for next ride along and land in the cache: the best-scoring unvisited
    // alternatives at every level of the path just walked, and the best-prior children of the nodes expanded before (where
    // the next visit of such a node goes: all its children have n = 0, so select takes the largest prior).  Nobody is parked
    // on those rows -- finish_batch only stores them -- and the cache returns exactly what a fresh evaluation returns (the
    // evaluator is batch invariant), so every search is unchanged; only the number of round trips is.
    //
    // Appends up to `budget` candidates of slot `s` to its evaluator's pending batch; returns how many were added.
    uint32_t add_speculative_rows(Slot& s, Group& gr, uint32_t budget) {
        Evaluator& ev = *evals_[s.cur];
        if (!budget || !ev.cache) return 0;
        Player& pl = s.players[s.cur];
        TreeT& t = pl.tree;
        Pending& pb = gr.pend[evals_[0] == evals_[1] ? 0 : s.cur];
        if (pb.keys.empty()) return 0;
        uint32_t added = 0;
        size_t sim_next = 0;
        // every level's best alternative before any level's second best
        std::stable_sort(s.sim_cands.begin(), s.sim_cands.end(), [](const SimCand& a, const SimCand& b) { return a.rank < b.rank; });
        while (added < budget && (sim_next < s.sim_cands.size() || pl.spec_head < pl.spec_queue.size())) {
            std::pair<int32_t, int32_t> cand;
            if (sim_next < s.sim_cands.size()) {
                cand = {s.sim_cands[sim_next].node, s.sim_cands[sim_next].child};
                ++sim_next;
            } else {
                cand = pl.spec_queue[pl.spec_head++];
            }
            if (TreeT::edge_child(t.edge(cand.first)[cand.second]) >= 0) continue;  // visited in the meantime
            if (add_row_ahead(t.hdr(cand.first).pos, move_at(t, cand.first, cand.second), pb, *ev.cache)) ++added;
        }
        s.sim_cands.erase(s.sim_cands.begin(), s.sim_cands.begin() + static_cast<std::ptrdiff_t>(sim_next));
        c_.speculative += added;
        if (pl.spec_head == pl.spec_queue.size()) {
            pl.spec_queue.clear();
            pl.spec_head = 0;
        }
        return added;
    }

    // The position after `m` in `parent` as one more row of `pb`, unless it is finished, cached or already in the batch.
    bool add_row_ahead(const Pos& parent, Move m, Pending& pb, Cache& cache) {
        if constexpr (kChess) {
            Pos child = R.moved(parent, m);
            Move buf[256];
            const int n = R.children(child, buf);
            if (n == 0) return false;  // a finished position is never evaluated
            uint64_t q[4];
            R.key_planes(child, q);
            const PosKey key{static_cast<u128>(q[0]) | (static_cast<u128>(q[1]) << 64), static_cast<u128>(q[2]) | (static_cast<u128>(q[3]) << 64)};
            if (cache.find(key, n, val_.data())) return false;
            if (pb.find_or_reserve(key) >= 0) return false;
            pb.keys.push_back(key);
            uint64_t pl[Rules::kPlanes];
            R.planes(child, pl);
            pb.planes.insert(pb.planes.end(), pl, pl + Rules::kPlanes);
            const size_t at = pb.legal.size();
            pb.legal.resize(at + Rules::kLegalBytes, 0);
            for (int k = 0; k < n; ++k) {
                const int idx = R.nn_idx(buf[k]);
                pb.legal[at + (idx >> 3)] |= static_cast<uint8_t>(1u << (idx & 7));
            }
            pb.n_legal.push_back(static_cast<uint8_t>(n));
            return true;
        } else {
            const Pos child = R.moved(parent, m);
            if (R.status(child) != 0) return false;
            const Pos view = child.turn != 1 ? R.flipped_boards(child) : child;  // NNetwork::evaluate's flip (net/mod.rs:74-87)
            const int n = popcount128(R.legal_mask(view));
            const PosKey key = R.key(view);
            if (cache.find(key, n, val_.data())) return false;
            if (pb.find_or_reserve(key) >= 0) return false;
            pb.keys.push_back(key);
            u128 pl[3];
            R.planes(view, pl);
            for (int c = 0; c < 3; ++c)
                for (int k = 0; k < abi_wpp_; ++k) pb.planes.push_back(static_cast<uint64_t>(pl[c] >> (64 * k)));
            pb.n_legal.push_back(static_cast<uint8_t>(n));
            return true;
        }
    }

    // Self-play: a group whose batch is far below the size up to which the device time is flat takes speculative rows from
    // the games parked on it (the trainer-sized job: a hundred games over a few threads).
    void fill_small_batches(Group& gr) {
        for (int e = 0; e < 2; ++e) {
            Pending& pb = gr.pend[e];
            const uint32_t real = static_cast<uint32_t>(pb.keys.size());
            const uint32_t target = std::min(kSpecTargetRows, evals_[e]->max_rows);
            if (real == 0 || real >= target) continue;
            uint32_t budget = target - real;
            const uint32_t per_game = std::min<uint32_t>(speculate_, std::max<uint32_t>(1, budget / static_cast<uint32_t>(pb.parked.size())));
            for (uint32_t si : pb.parked) {
                if (!budget) break;
                budget -= add_speculative_rows(slots_[si], gr, std::min(per_game, budget));
            }
        }
    }

    // ---------------------------------------------------------------- evaluator batch
    static const uint8_t* legal_ptr(const Pending& pb) { return kChess ? pb.legal.data() : nullptr; }
    // Ship group `gr`'s batch for evaluator `e`: asynchronously when the evaluator supports it (collected at the
    // group's next turn), else evaluated and delivered on the spot.
    void send(Group& gr, int e) {
        Pending& pb = gr.pend[e];
        Evaluator& ev = *evals_[e];
        const uint32_t n = static_cast<uint32_t>(pb.keys.size());
        if (ev.async_handle && !(n == 1 && ev.leaf_handle) && n <= ev.max_rows) {  // larger than one device batch: the synchronous call below chunks
            const auto t0 = Clock::now();
            int32_t ticket = -1;
            int rc = cattus_b200_eval_batch_submit(ev.async_handle, pb.planes.data(), legal_ptr(pb), n, 0, &ticket);
            while (rc == 0 && ticket < 0) {
                // Every stream is busy.  Take back our own oldest batch (its results go to its games right away) and try
                // again; a worker only ever BLOCKS for a stream while holding none, so workers cannot deadlock each other.
                if (inflight_.empty()) {
                    rc = cattus_b200_eval_batch_submit(ev.async_handle, pb.planes.data(), legal_ptr(pb), n, 1, &ticket);
                    break;
                }
                const std::pair<uint32_t, int> oldest = inflight_.front();
                collect(groups_[oldest.first], oldest.second);
                rc = cattus_b200_eval_batch_submit(ev.async_handle, pb.planes.data(), legal_ptr(pb), n, 0, &ticket);
            }
            eval_wait_ += std::chrono::duration<double>(Clock::now() - t0).count();
            if (rc != 0) throw SpError{rc, std::string("evaluator failed: ") + cattus_b200_last_error()};
            gr.ticket[e] = ticket;
            gr.inflight_n[e] = n;
            inflight_.emplace_back(static_cast<uint32_t>(&gr - groups_.data()), e);
            return;
        }
        size_t total = 0;
        for (uint8_t c : pb.n_legal) total += c;
        probs_.resize(total);
        offsets_.resize(n + 1);
        values_.resize(n);
        const auto t0 = Clock::now();
        int rc;
        if (n == 1 && ev.leaf_handle) {
            uint32_t np = 0;
            rc = cattus_b200_eval(ev.leaf_handle, pb.planes.data(), legal_ptr(pb), probs_.data(), static_cast<uint32_t>(total), &np, values_.data());
            offsets_[0] = 0;
            offsets_[1] = np;
        } else {
            rc = ev.fn(ev.ctx, pb.planes.data(), legal_ptr(pb), n, probs_.data(), total, offsets_.data(), values_.data());
        }
        eval_wait_ += std::chrono::duration<double>(Clock::now() - t0).count();
        if (rc != 0) throw SpError{rc, std::string("evaluator failed: ") + cattus_b200_last_error()};
        finish_batch(pb, ev, n);
    }

    // Wait for group `gr`'s batch in flight on evaluator `e` and hand the results to its parked games.
    void collect(Group& gr, int e) {
        Pending& pb = gr.pend[e];
        Evaluator& ev = *evals_[e];
        const uint32_t n = gr.inflight_n[e];
        size_t total = 0;
        for (uint8_t c : pb.n_legal) total += c;
        probs_.resize(total);
        offsets_.resize(n + 1);
        values_.resize(n);
        const auto t0 = Clock::now();
        const int rc = cattus_b200_eval_batch_wait(ev.async_handle, gr.ticket[e], probs_.data(), total, offsets_.data(), values_.data());
        eval_wait_ += std::chrono::duration<double>(Clock::now() - t0).count();
        gr.ticket[e] = -1;
        const std::pair<uint32_t, int> me(static_cast<uint32_t>(&gr - groups_.data()), e);
        inflight_.erase(std::find(inflight_.begin(), inflight_.end(), me));
        if (rc != 0) throw SpError{rc, std::string("evaluator failed: ") + cattus_b200_last_error()};
        finish_batch(pb, ev, n);
    }

    // error / shutdown path: every submitted ticket must be waited exactly once
    void drain_all() {
        for (Group& gr : groups_)
            for (int e = 0; e < 2; ++e)
                if (gr.ticket[e] >= 0) {
                    Pending& pb = gr.pend[e];
                    size_t total = 0;
                    for (uint8_t c : pb.n_legal) total += c;
                    probs_.resize(total);
                    offsets_.resize(gr.inflight_n[e] + 1);
                    values_.resize(gr.inflight_n[e]);
                    cattus_b200_eval_batch_wait(evals_[e]->async_handle, gr.ticket[e], probs_.data(), total, offsets_.data(), values_.data());
                    gr.ticket[e] = -1;
                }
        inflight_.clear();
    }

    // rows -> (probs..., value), through the cache (cache.rs:44-73), then to the games parked on this batch
    void finish_batch(Pending& pb, Evaluator& ev, uint32_t n) {
        c_.batches += 1;
        c_.evaluations += n;
        const size_t stride = val_.size();
        rows_.resize(static_cast<size_t>(n) * stride);
        for (uint32_t r = 0; r < n; ++r) {
            const uint32_t cnt = pb.n_legal[r];
            if (offsets_[r + 1] - offsets_[r] != cnt) throw SpError{CATTUS_B200_EINVAL, "evaluator returned a wrong number of probabilities"};
            float* v = rows_.data() + r * stride;
            std::memcpy(v, probs_.data() + offsets_[r], sizeof(float) * cnt);
            v[cnt] = values_[r];
            if (ev.cache) {
                if (ev.cache->insert(pb.keys[r], static_cast<int>(cnt), v))
                    c_.cache_misses += 1;
                else
                    c_.cache_hits += 1;
            }
        }
        for (uint32_t si : pb.parked) {
            Slot& s = slots_[si];
            deliver(s, rows_.data() + s.wait_row * stride);
            s.phase = kSimulate;
        }
        pb.clear();
    }

    const Rules& R;
    const cattus_b200_selfplay_cfg& cfg_;
    Shared& sh_;
    Params params_[2];
    Evaluator* evals_[2];
    std::vector<Slot> slots_;
    std::vector<Group> groups_;
    std::vector<std::vector<uint32_t>> pool_free_;  // retired tree buffers, reused by the next tree copy
    uint32_t speculate_ = 0;  // rows evaluated ahead per game and evaluator call (cfg.speculate)
    static constexpr uint32_t kSpecTargetRows = 192;  // batches below this take speculative rows (device time is flat to ~256)
    static constexpr int kSpecPerLevel = 4;
    std::deque<std::pair<uint32_t, int>> inflight_;  // (group, evaluator) of this worker's batches in flight, oldest first
    int abi_wpp_ = 1;
    double eval_wait_ = 0.0;
    std::vector<double> noise_;
    std::vector<float> weights_, probs_, values_, val_, rows_;
    float sel_[256];  // selection values of one node's children (<= 121 cells, <= 218 chess moves)
    static constexpr uint32_t kMaxRing = 32;
    uint32_t ring_size_ = 8;  // games advanced interleaved (memory-level parallelism of the tree walks); CATTUS_B200_SELFPLAY_RING
    Counters c_;
    std::vector<uint32_t> offsets_;
};

static void make_dirs(const char* path) {
    std::string p(path);
    for (size_t i = 1; i <= p.size(); ++i)
        if (i == p.size() || p[i] == '/') {
            const std::string sub = p.substr(0, i);
            ::mkdir(sub.c_str(), 0777);
        }
}

}  // namespace sp

struct cattus_b200_selfplay {
    cattus_b200_selfplay_summary summary;
    uint64_t minibatches = 0, collisions = 0;
    std::vector<sp::GameRecord> records;
};

static thread_local std::string g_sp_error;

template <class Rules>
static void run_games(const Rules& rules, const cattus_b200_selfplay_cfg& cfg, const sp::Params params[2], sp::Evaluator* evals[2], sp::Shared& sh) {
    const uint32_t n_threads = std::max<uint32_t>(1, cfg.threads);
    std::vector<std::unique_ptr<sp::Worker<Rules>>> workers;
    for (uint32_t i = 0; i < n_threads; ++i) workers.emplace_back(new sp::Worker<Rules>(rules, cfg, params, evals, sh));
    struct Joiner {  // joins on every exit path: an exception on the calling thread must not destroy joinable threads
        std::vector<std::thread> threads;
        ~Joiner() {
            for (auto& t : threads)
                if (t.joinable()) t.join();
        }
    } joiner;
    for (uint32_t i = 1; i < n_threads; ++i) joiner.threads.emplace_back([&, i] { workers[i]->run(); });
    workers[0]->run();  // the calling thread does job 0 (self_play.rs:127-137); run() itself never throws
}

static int selfplay_impl(sp::Evaluator& e1, sp::Evaluator* e2_or_null, const cattus_b200_selfplay_cfg* cfg, cattus_b200_selfplay_t** out,
                         const cattus_b200_selfplay_opts* opts = nullptr) {
    try {
        if (!cfg || !out) throw sp::SpError{CATTUS_B200_EINVAL, "null argument"};
        if (cfg->struct_size != sizeof(cattus_b200_selfplay_cfg)) throw sp::SpError{CATTUS_B200_EINVAL, "selfplay cfg struct_size mismatch"};
        *out = nullptr;
        const uint32_t L = sp::selfplay_search_batch(opts, *cfg);
        const uint32_t search_batch[2] = {L, L};
        if (cfg->games_num % 2 != 0) throw sp::SpError{CATTUS_B200_EINVAL, "Games num should be a multiple of 2 (self_play.rs:100)"};
        if ((cfg->out_dir1 == nullptr) != (cfg->out_dir2 == nullptr)) throw sp::SpError{CATTUS_B200_EINVAL, "out_dir1 and out_dir2 must both be set or both NULL"};
        const sp::Params p = sp::parse_params(cfg);
        sp::Params params[2] = {p, p};
        if (cfg->game == CATTUS_B200_GAME_HEX) {
            if (cfg->board_size < 2 || cfg->board_size > 11) throw sp::SpError{CATTUS_B200_EINVAL, "hex board_size must be 2..11"};
        } else if (cfg->game != CATTUS_B200_GAME_TTT && cfg->game != CATTUS_B200_GAME_CHESS) {
            throw sp::SpError{CATTUS_B200_EINVAL, "unknown game"};
        }
        if (cfg->cache_size && !cfg->device_games) {
            // room per entry: the most legal moves a position can have, plus the value
            const int moves_num = cfg->game == CATTUS_B200_GAME_TTT     ? 9
                                  : cfg->game == CATTUS_B200_GAME_CHESS ? sp::ChessRules::kMaxMoves
                                                                        : static_cast<int>(cfg->board_size * cfg->board_size);
            e1.cache.reset(new sp::Cache(cfg->cache_size, moves_num));
            if (e2_or_null) e2_or_null->cache.reset(new sp::Cache(cfg->cache_size, moves_num));
        }
        sp::Evaluator* evals[2] = {&e1, e2_or_null ? e2_or_null : &e1};
        if (cfg->out_dir1) {
            sp::make_dirs(cfg->out_dir1);
            sp::make_dirs(cfg->out_dir2);
        }
        sp::Shared sh;
        const auto t0 = sp::Clock::now();
        if (cfg->device_games) {
            // trees in HBM, one warp per game (dsearch_core.hpp): needs the B200 evaluator's device buffers
            if (!e1.async_handle || (e2_or_null && !e2_or_null->async_handle))
                throw sp::SpError{CATTUS_B200_EINVAL, "device_games needs the B200 evaluator (cattus_b200_selfplay_run); a callback evaluator has no device buffers"};
            cb2::dsearch_run(e1.async_handle, e2_or_null ? e2_or_null->async_handle : nullptr, *cfg, params, search_batch, sh);
        } else if (cfg->game == CATTUS_B200_GAME_HEX) {
            if (cfg->board_size <= 8) {
                sp::HexRulesT<uint64_t> rules(static_cast<int>(cfg->board_size));
                run_games(rules, *cfg, params, evals, sh);
            } else {
                sp::HexRulesT<sp::u128> rules(static_cast<int>(cfg->board_size));
                run_games(rules, *cfg, params, evals, sh);
            }
        } else if (cfg->game == CATTUS_B200_GAME_CHESS) {
            sp::ChessRules rules;
            run_games(rules, *cfg, params, evals, sh);
        } else {
            sp::TttRules rules;
            run_games(rules, *cfg, params, evals, sh);
        }
        if (sh.failed.load()) throw sp::SpError{sh.error_code, sh.error};
        std::unique_ptr<cattus_b200_selfplay> r(new cattus_b200_selfplay());
        cattus_b200_selfplay_summary& s = r->summary;
        std::memset(&s, 0, sizeof(s));
        s.player1_wins = sh.w1;
        s.player2_wins = sh.w2;
        s.draws = sh.d;
        s.games = sh.games;
        s.simulations = sh.simulations;
        s.searches = sh.searches;
        s.evaluations = sh.evaluations;
        s.cache_hits = sh.cache_hits;
        s.cache_misses = sh.cache_misses;
        s.batches = sh.batches;
        s.terminal_leaves = sh.terminal;
        s.seconds = std::chrono::duration<double>(sp::Clock::now() - t0).count();
        s.search_duration = sh.search_duration;
        s.eval_wait_seconds = sh.eval_wait;
        s.speculative_evaluations = sh.speculative;
        // the host-tree driver keeps one leaf in flight: a round per simulation
        r->minibatches = cfg->device_games ? sh.minibatches[0] + sh.minibatches[1] : sh.simulations;
        r->collisions = sh.collisions[0] + sh.collisions[1];
        r->records = std::move(sh.records);
        std::sort(r->records.begin(), r->records.end(), [](const sp::GameRecord& a, const sp::GameRecord& b) { return a.game_idx < b.game_idx; });
        *out = r.release();
        g_sp_error.clear();
        return CATTUS_B200_OK;
    } catch (const sp::SpError& e) {
        g_sp_error = e.msg;
        return e.code ? e.code : CATTUS_B200_EINVAL;
    } catch (const std::exception& e) {
        g_sp_error = e.what();
        return CATTUS_B200_EINVAL;
    }
}

static uint32_t handle_max_batch(const cattus_b200_t* h) {
    cattus_b200_info info;
    return cattus_b200_get_info(h, &info) == CATTUS_B200_OK && info.max_batch ? info.max_batch : 1u;
}

static int engine_eval_thunk(void* ctx, const uint64_t* planes, const uint8_t* legal, uint32_t n, float* probs, size_t cap, uint32_t* offsets, float* values) {
    return cattus_b200_eval_batch(static_cast<cattus_b200_t*>(ctx), planes, legal, n, probs, cap, offsets, values);
}

extern "C" {

int cattus_b200_selfplay_run(cattus_b200_t* model1, cattus_b200_t* model2, const cattus_b200_selfplay_cfg* cfg, cattus_b200_selfplay_t** out) {
    return cattus_b200_selfplay_run_opts(model1, model2, cfg, nullptr, out);
}

int cattus_b200_selfplay_run_opts(cattus_b200_t* model1, cattus_b200_t* model2, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_selfplay_opts* opts,
                                  cattus_b200_selfplay_t** out) {
    if (!model1) {
        g_sp_error = "null evaluator handle (there is no CPU fallback)";
        return CATTUS_B200_EINVAL;
    }
    sp::Evaluator e1, e2;
    e1.fn = engine_eval_thunk;
    e1.ctx = model1;
    e1.async_handle = model1;
    e1.max_rows = handle_max_batch(model1);
    if (cfg && cfg->leaf_queue) e1.leaf_handle = model1;
    const bool two = model2 && model2 != model1;
    if (two) {
        e2.fn = engine_eval_thunk;
        e2.ctx = model2;
        e2.async_handle = model2;
        e2.max_rows = handle_max_batch(model2);
        if (cfg && cfg->leaf_queue) e2.leaf_handle = model2;
    }
    return selfplay_impl(e1, two ? &e2 : nullptr, cfg, out, opts);
}

int cattus_b200_selfplay_run_with(cattus_b200_eval_fn eval1, void* ctx1, cattus_b200_eval_fn eval2, void* ctx2, const cattus_b200_selfplay_cfg* cfg,
                                  cattus_b200_selfplay_t** out) {
    if (!eval1) {
        g_sp_error = "null evaluator callback";
        return CATTUS_B200_EINVAL;
    }
    sp::Evaluator e1, e2;
    e1.fn = eval1;
    e1.ctx = ctx1;
    const bool two = eval2 && !(eval2 == eval1 && ctx2 == ctx1);
    if (two) {
        e2.fn = eval2;
        e2.ctx = ctx2;
    }
    return selfplay_impl(e1, two ? &e2 : nullptr, cfg, out);
}

int cattus_b200_selfplay_summary_get(const cattus_b200_selfplay_t* r, cattus_b200_selfplay_summary* out) {
    if (!r || !out) return CATTUS_B200_EINVAL;
    *out = r->summary;
    return CATTUS_B200_OK;
}

int cattus_b200_selfplay_batches(const cattus_b200_selfplay_t* r, uint64_t* minibatches, uint64_t* collisions) {
    if (!r) return CATTUS_B200_EINVAL;
    if (minibatches) *minibatches = r->minibatches;
    if (collisions) *collisions = r->collisions;
    return CATTUS_B200_OK;
}

int cattus_b200_selfplay_game_count(const cattus_b200_selfplay_t* r, uint32_t* n) {
    if (!r || !n) return CATTUS_B200_EINVAL;
    *n = static_cast<uint32_t>(r->records.size());
    return CATTUS_B200_OK;
}

int cattus_b200_selfplay_game_info(const cattus_b200_selfplay_t* r, uint32_t k, uint32_t* game_idx, uint32_t* winner, uint32_t* n_moves) {
    if (!r || k >= r->records.size()) return CATTUS_B200_ERANGE;
    if (game_idx) *game_idx = r->records[k].game_idx;
    if (winner) *winner = r->records[k].winner;
    if (n_moves) *n_moves = static_cast<uint32_t>(r->records[k].moves.size());
    return CATTUS_B200_OK;
}

int cattus_b200_selfplay_game_moves(const cattus_b200_selfplay_t* r, uint32_t k, uint8_t* moves_out, uint32_t cap) {
    if (!r || !moves_out || k >= r->records.size()) return CATTUS_B200_ERANGE;
    const auto& m = r->records[k].moves;
    if (cap < m.size()) return CATTUS_B200_ERANGE;
    for (size_t i = 0; i < m.size(); ++i) {
        if (m[i] > 0xFF) return CATTUS_B200_ERANGE;  // chess moves need cattus_b200_selfplay_game_moves16
        moves_out[i] = static_cast<uint8_t>(m[i]);
    }
    return CATTUS_B200_OK;
}

int cattus_b200_selfplay_game_moves16(const cattus_b200_selfplay_t* r, uint32_t k, uint16_t* moves_out, uint32_t cap) {
    if (!r || !moves_out || k >= r->records.size()) return CATTUS_B200_ERANGE;
    const auto& m = r->records[k].moves;
    if (cap < m.size()) return CATTUS_B200_ERANGE;
    std::memcpy(moves_out, m.data(), m.size() * sizeof(uint16_t));
    return CATTUS_B200_OK;
}

int cattus_b200_selfplay_entry(const cattus_b200_selfplay_t* r, uint32_t k, uint32_t pos_idx, uint8_t* bytes_out, size_t cap, size_t* n_bytes,
                               uint32_t* out_dir) {
    if (!r || k >= r->records.size() || pos_idx >= r->records[k].entries.size()) return CATTUS_B200_ERANGE;
    const auto& b = r->records[k].entries[pos_idx];
    if (n_bytes) *n_bytes = b.size();
    if (out_dir) *out_dir = r->records[k].entry_dir[pos_idx];
    if (bytes_out) {
        if (cap < b.size()) return CATTUS_B200_ERANGE;
        std::memcpy(bytes_out, b.data(), b.size());
    }
    return CATTUS_B200_OK;
}

void cattus_b200_selfplay_free(cattus_b200_selfplay_t* r) { delete r; }

// ---------------------------------------------------------------- one chess search at a time (the UCI loop's player)
struct cattus_b200_chess_search {
    sp::ChessRules rules;
    cattus_b200_selfplay_cfg cfg;
    sp::Params params[2];
    sp::Evaluator ev;
    sp::Evaluator* evals[2];
    sp::Shared sh;
    std::unique_ptr<sp::Worker<sp::ChessRules>> worker;
};

static int chess_search_create_impl(cattus_b200_eval_fn fn, void* ctx, cattus_b200_t* leaf_handle, const cattus_b200_selfplay_cfg* cfg,
                                    cattus_b200_chess_search_t** out) {
    try {
        if (!cfg || !out || !fn) throw sp::SpError{CATTUS_B200_EINVAL, "null argument"};
        if (cfg->struct_size != sizeof(cattus_b200_selfplay_cfg)) throw sp::SpError{CATTUS_B200_EINVAL, "selfplay cfg struct_size mismatch"};
        *out = nullptr;
        std::unique_ptr<cattus_b200_chess_search> s(new cattus_b200_chess_search());
        s->params[0] = s->params[1] = sp::parse_params(cfg);
        s->cfg = *cfg;
        s->cfg.game = CATTUS_B200_GAME_CHESS;
        s->cfg.board_size = 8;
        s->cfg.temperature_moves = nullptr;  // consumed by parse_params; the caller's arrays need not outlive this call
        s->cfg.temperature_values = nullptr;
        s->cfg.threads = s->cfg.games_per_thread = 1;
        s->cfg.groups_per_thread = s->cfg.keep_records = s->cfg.max_moves = s->cfg.first_game = 0;
        s->cfg.game_stride = 1;
        s->cfg.games_num = 2;
        s->cfg.out_dir1 = s->cfg.out_dir2 = nullptr;
        s->ev.fn = fn;
        s->ev.ctx = ctx;
        s->ev.leaf_handle = leaf_handle;
        if (leaf_handle) s->ev.max_rows = handle_max_batch(leaf_handle);
        // One tree fills the table slowly (<= sim_num entries per search), and every entry of a table sized for a million
        // positions would land on a fresh page: most of a search's host time went into page faults.  128 Ki entries hold the
        // last dozen searches; a smaller cache only changes hit rates, never results.
        if (cfg->cache_size) s->ev.cache.reset(new sp::Cache(std::min<uint32_t>(cfg->cache_size, 1u << 17), sp::ChessRules::kMaxMoves));
        s->evals[0] = s->evals[1] = &s->ev;
        s->worker.reset(new sp::Worker<sp::ChessRules>(s->rules, s->cfg, s->params, s->evals, s->sh));
        s->worker->reseed(cfg->seed);
        s->worker->set_speculation(cfg->speculate);
        *out = s.release();
        g_sp_error.clear();
        return CATTUS_B200_OK;
    } catch (const sp::SpError& e) {
        g_sp_error = e.msg;
        return e.code ? e.code : CATTUS_B200_EINVAL;
    } catch (const std::exception& e) {
        g_sp_error = e.what();
        return CATTUS_B200_EINVAL;
    }
}

int cattus_b200_chess_search_create(cattus_b200_t* model, const cattus_b200_selfplay_cfg* cfg, cattus_b200_chess_search_t** out) {
    if (!model) {
        g_sp_error = "null evaluator handle (there is no CPU fallback)";
        return CATTUS_B200_EINVAL;
    }
    return chess_search_create_impl(engine_eval_thunk, model, model, cfg, out);
}

int cattus_b200_chess_search_create_with(cattus_b200_eval_fn eval, void* ctx, const cattus_b200_selfplay_cfg* cfg, cattus_b200_chess_search_t** out) {
    return chess_search_create_impl(eval, ctx, nullptr, cfg, out);
}

int cattus_b200_chess_search_go(cattus_b200_chess_search_t* s, const char* fen, const uint16_t* moves, uint32_t n_moves, uint16_t* best_move,
                                cattus_b200_chess_search_stats* stats) {
    try {
        if (!s || !best_move || (n_moves && !moves)) throw sp::SpError{CATTUS_B200_EINVAL, "null argument"};
        const sp::ChessRules& R = s->rules;
        std::vector<sp::ChessPos> history;
        sp::ChessPos p;
        if (fen) {
            const std::string err = R.from_fen(fen, p);
            if (!err.empty()) throw sp::SpError{CATTUS_B200_EINVAL, "bad FEN: " + err};
        } else {
            p = R.initial();
        }
        history.push_back(p);
        sp::ChessRules::Move buf[256];
        for (uint32_t i = 0; i < n_moves; ++i) {  // cmd_position (uci.rs:76-93): moved_position per move, every position kept
            const int n = R.children(p, buf);
            const sp::ChessRules::Move want = sp::ChessRules::real_move(p, moves[i]);
            bool found = false;
            for (int k = 0; k < n; ++k) found |= buf[k] == want;
            if (!found) throw sp::SpError{CATTUS_B200_EINVAL, "move " + std::to_string(i) + " is not legal here"};
            p = R.moved(p, want);
            R.children(p, buf);  // settles status()
            history.push_back(p);
        }
        sp::Worker<sp::ChessRules>::SearchStats st;
        sp::ChessRules::Move best = 0;
        if (!s->worker->search_from(history, &best, &st)) {
            if (s->sh.failed.load()) throw sp::SpError{s->sh.error_code, s->sh.error};
            throw sp::SpError{CATTUS_B200_EINVAL, "the game is over in this position: no move to search"};
        }
        *best_move = best;
        if (stats) {
            if (stats->struct_size != sizeof(cattus_b200_chess_search_stats)) throw sp::SpError{CATTUS_B200_EINVAL, "search stats struct_size mismatch"};
            stats->simulations = st.simulations;
            stats->evaluations = st.evaluations;
            stats->cache_hits = st.cache_hits;
            stats->terminal_leaves = st.terminal;
            stats->seconds = st.seconds;
            stats->root_children = st.root_children;
            stats->best_visits = st.root_visits_best;
            stats->speculative_evaluations = st.speculative;
        }
        g_sp_error.clear();
        return CATTUS_B200_OK;
    } catch (const sp::SpError& e) {
        g_sp_error = e.msg;
        return e.code ? e.code : CATTUS_B200_EINVAL;
    } catch (const std::exception& e) {
        g_sp_error = e.what();
        return CATTUS_B200_EINVAL;
    }
}

void cattus_b200_chess_search_destroy(cattus_b200_chess_search_t* s) { delete s; }

const char* cattus_b200_selfplay_last_error(void) { return g_sp_error.c_str(); }

}  // extern "C"
