// Host half of the batched analysis of given positions on the device-resident search (the per-simulation half is the
// same dsearch_core.hpp that self-play runs).
//
// Self-play hands every slot a game and answers each finished search with the next move; analysis hands every slot a
// POSITION: one kCmdSetRoot command installs the position with its history as a fresh tree, the slot runs sim_num
// simulations, and the device posts the root rows and the principal variation (Params::analysis).  The driver stores
// them under the position's input index and gives the slot the next position.  Each position is searched as a fresh
// MctsPlayer (engine/src/mcts/mod.rs:335-385) searches it with no root noise: no tree is kept between positions, so a
// result depends neither on the number of slots, the waves in flight, the cache nor where the position falls in the input.
//
// `Backend` is the self-play transport (dsearch.cuh's DsCudaBackend, tests/emul's emulation) built with the analysis
// result layout and a root upload: roots_block(wave) / roots_cap() is where a wave's root histories are staged before
// submit() uploads them.
#pragma once

#include <deque>
#include <string>
#include <vector>

#include "../../include/cattus_b200_analysis.h"
#include "dsearch_core.hpp"
#include "dsearch_host.hpp"
#include "sp_common.hpp"

namespace ds {

struct AnalysisOpts {
    uint32_t pv_max;  // principal variation plies (<= kPvMax)
};

// A minibatched search's entry ends in 16 more bytes: u32 minibatches, u32 collisions (batch_expand_slot).
inline uint32_t analysis_stride_for(uint32_t max_children, uint32_t search_batch = 1) {
    return ((static_cast<uint32_t>(sizeof(AnalysisHdr)) + 2u * kPvMax + 14u * max_children + 15u) & ~15u) + (search_batch > 1 ? 16u : 0u);
}

// search_batch of the C ABI's options: NULL, 0 or 1 is one leaf in flight.
inline uint32_t analysis_search_batch(const cattus_b200_analysis_opts* opts) {
    if (!opts) return 1;
    if (opts->struct_size != sizeof(cattus_b200_analysis_opts)) throw sp::SpError{CATTUS_B200_EINVAL, "analysis opts struct_size mismatch"};
    return opts->search_batch ? opts->search_batch : 1u;
}

// Concurrent searches of an analysis of n positions, or of a match of n games: device_games, 0 = min(n, max_batch /
// search_batch).  Every slot writes up to search_batch evaluator rows per wave (a match: the larger side's), so
// device_games x search_batch above max_batch is ERANGE.
inline uint32_t analysis_slots(uint32_t device_games, uint32_t n, uint32_t max_batch, uint32_t search_batch) {
    if (search_batch > 1 && static_cast<uint64_t>(device_games ? device_games : 1u) * search_batch > max_batch)
        throw sp::SpError{CATTUS_B200_ERANGE, "device search: device_games (" + std::to_string(device_games) + ") x search_batch (" +
                                                  std::to_string(search_batch) + ") exceeds the evaluator's max_batch (" + std::to_string(max_batch) + ")"};
    if (device_games > max_batch)
        throw sp::SpError{CATTUS_B200_ERANGE, "device search: device_games (" + std::to_string(device_games) + ") exceeds the evaluator's max_batch (" +
                                                  std::to_string(max_batch) + ")"};
    const uint32_t want = device_games ? device_games : max_batch / search_batch;
    return std::max<uint32_t>(1, std::min<uint32_t>(want, n));
}

// Concurrent games of a self-play partition of `games` games (device_games > 0): with minibatches (search_batch > 1)
// checked as analysis_slots checks them; with one leaf in flight the backend checks the slots against max_batch.
inline uint32_t selfplay_slots(uint32_t device_games, uint32_t games, uint32_t max_batch, uint32_t search_batch) {
    if (search_batch > 1) return analysis_slots(device_games, games, max_batch, search_batch);
    return std::max<uint32_t>(1, std::min<uint32_t>(device_games, games));
}

// The history ring of a slot (dsearch.cuh allocates it): chess keeps what detect_repetition can look back into, the
// other games only the root.
template <class Rules>
constexpr uint32_t hist_cap_for() {
    return Rules::kChess ? 128u : 1u;
}

// One analysed position.  Children in edges() order (newest first), the order calc_moves_probabilities returns them;
// moves in the game's real encoding (chess: from | to << 6 | promotion << 12 in real board coordinates; hex and
// tic-tac-toe: cell index).
struct AnalysisResult {
    uint32_t status = 0;       // 0: searched; 1 / 2: finished, that player won; 3: draw (also threefold repetition) -- not searched
    uint32_t simulations = 0;  // develop_tree iterations of the search
    uint16_t best = 0;         // choose_move_from_probabilities at temperature 0 over the visit distribution
    float q = 0.0f;            // sum W / sum N over the root's children: the side to move's mean score in [-1, 1]
    std::vector<uint16_t> moves;
    std::vector<uint32_t> visits;
    std::vector<float> w, prior;
    std::vector<uint16_t> pv;
    uint32_t minibatches = 0;  // rounds of descents (one leaf in flight: one per simulation)
    uint32_t collisions = 0;   // descents that ended on a leaf an earlier descent of their minibatch had claimed
    // a session's search (dsearch_session.hpp): the root's visits kept from the previous search, why it ended
    // (cattus_b200_session.h's CATTUS_B200_STOP_*) and its seconds; zero elsewhere
    uint32_t reused = 0, stop_reason = 0;
    double seconds = 0.0;
};

// a move of the device's tree in the game's real encoding (chess trees hold the side to move's view)
template <class Rules>
uint16_t analysis_real_move(const typename Rules::Pos& p, uint32_t m) {
    if constexpr (Rules::kChess)
        return Rules::real_move(p, static_cast<typename Rules::Move>(m));
    else
        return static_cast<uint16_t>(m);
}

// Fills `r` from a posted analysis entry `e` of the search of `root` (count and pv_len already checked): the children in
// edges() order, the best move, q and the principal variation; with minibatches (search_batch > 1) the entry's counts.
template <class Rules>
void read_analysis_entry(const Rules& R, const sp::Params& params, const typename Rules::Pos& root, const uint8_t* e, uint32_t maxc,
                         uint32_t result_stride, uint32_t search_batch, AnalysisResult& r,
                         std::vector<std::pair<typename Rules::Move, float>>& probs, std::vector<float>& weights) {
    using Pos = typename Rules::Pos;
    using Move = typename Rules::Move;
    const AnalysisHdr* ah = reinterpret_cast<const AnalysisHdr*>(e);
    const uint32_t count = ah->count, pv_len = ah->pv_len;
    const uint16_t* pv = reinterpret_cast<const uint16_t*>(e + sizeof(AnalysisHdr));
    const uint32_t* rn = reinterpret_cast<const uint32_t*>(e + sizeof(AnalysisHdr) + 2u * kPvMax);
    const float* rw = reinterpret_cast<const float*>(rn + maxc);
    const float* ri = rw + maxc;
    const uint16_t* rm = reinterpret_cast<const uint16_t*>(ri + maxc);
    r.status = 0;
    r.simulations = params.sim_num;
    r.minibatches = params.sim_num;
    r.collisions = 0;
    if (search_batch > 1) {
        const uint32_t* counts = reinterpret_cast<const uint32_t*>(e + result_stride - 16u);
        r.minibatches = counts[0];
        r.collisions = counts[1];
    }
    uint32_t total = 0;
    double sw = 0.0;
    for (uint32_t i = 0; i < count; ++i) {
        total += rn[i];
        sw += static_cast<double>(rw[i]);
    }
    r.moves.clear();
    r.visits.clear();
    r.w.clear();
    r.prior.clear();
    r.pv.clear();
    probs.clear();
    for (int32_t i = static_cast<int32_t>(count) - 1; i >= 0; --i) {  // edges() order
        r.moves.push_back(analysis_real_move<Rules>(root, rm[i]));
        r.visits.push_back(rn[i]);
        r.w.push_back(rw[i]);
        r.prior.push_back(ri[i]);
        probs.emplace_back(static_cast<Move>(rm[i]), static_cast<float>(rn[i]) / static_cast<float>(total));
    }
    sp::SplitMix64 unused(0);
    r.best = r.moves[static_cast<size_t>(sp::choose_move(params, 0, probs, unused, weights))];
    r.q = total ? static_cast<float>(sw / static_cast<double>(total)) : 0.0f;
    Pos p = root;
    for (uint32_t j = 0; j < pv_len; ++j) {
        r.pv.push_back(analysis_real_move<Rules>(p, pv[j]));
        if (j + 1 < pv_len) p = R.moved(p, static_cast<Move>(pv[j]));
    }
}

// MctsParams of an analysis: the mcts.* fields without root noise (a noisy search would not be an analysis of the
// position, and its samples would depend on the order of the positions).
inline sp::Params analysis_params(const cattus_b200_selfplay_cfg& cfg) {
    if (cfg.struct_size != sizeof(cattus_b200_selfplay_cfg)) throw sp::SpError{CATTUS_B200_EINVAL, "selfplay cfg struct_size mismatch"};
    if (cfg.prior_noise_epsilon != 0.0f)
        throw sp::SpError{CATTUS_B200_EINVAL, "analysis: prior_noise_epsilon must be 0 (root noise is not part of an analysis)"};
    if (cfg.sim_num < 2) throw sp::SpError{CATTUS_B200_EINVAL, "analysis: sim_num must be > 1 (mcts/mod.rs:157)"};
    if (!(cfg.explore_factor >= 0.0f)) throw sp::SpError{CATTUS_B200_EINVAL, "analysis: explore_factor must be >= 0"};
    if (cfg.game == CATTUS_B200_GAME_HEX) {
        if (cfg.board_size < 2 || cfg.board_size > 11) throw sp::SpError{CATTUS_B200_EINVAL, "hex board_size must be 2..11"};
    } else if (cfg.game != CATTUS_B200_GAME_TTT && cfg.game != CATTUS_B200_GAME_CHESS) {
        throw sp::SpError{CATTUS_B200_EINVAL, "unknown game"};
    }
    sp::Params p;
    p.sim_num = cfg.sim_num;
    p.explore_factor = cfg.explore_factor;
    p.noise_alpha = 0.0f;
    p.noise_eps = 0.0f;
    p.last_temperature = 0.0f;  // the best move is the temperature-0 choice
    return p;
}

// Position k = fens[k] (NULL: the game's initial position; chess only otherwise) followed by moves[move_offsets[k],
// move_offsets[k + 1]).  Returns each position's history as far as the search can need it: for chess the positions
// since the last pawn move or capture (at most hist_cap_for), for the other games the position alone.  Every position
// has its status settled.  Errors name the input as `what` k ("position 3: ...").
template <class Rules>
std::vector<std::vector<typename Rules::Pos>> analysis_histories(const Rules& R, uint32_t n, const char* const* fens, const uint16_t* moves,
                                                                 const uint32_t* move_offsets, const char* what = "position") {
    using Pos = typename Rules::Pos;
    using Move = typename Rules::Move;
    std::vector<std::vector<Pos>> out(n);
    const auto fail = [what](uint32_t k, const std::string& why) {
        return sp::SpError{CATTUS_B200_EINVAL, std::string(what) + " " + std::to_string(k) + ": " + why};
    };
    for (uint32_t k = 0; k < n; ++k) {
        const uint32_t m0 = move_offsets ? move_offsets[k] : 0u, m1 = move_offsets ? move_offsets[k + 1] : 0u;
        if (m1 < m0) throw fail(k, "move_offsets decrease");
        if (m1 > m0 && !moves) throw fail(k, "moves is NULL");
        const char* fen = fens ? fens[k] : nullptr;
        std::vector<Pos>& h = out[k];
        Pos p;
        if constexpr (Rules::kChess) {
            Move buf[256];
            if (fen) {
                const std::string err = R.from_fen(fen, p);
                if (!err.empty()) throw fail(k, "bad FEN: " + err);
            } else {
                p = R.initial();
            }
            R.children(p, buf);  // settles status()
            h.push_back(p);
            for (uint32_t i = m0; i < m1; ++i) {
                const int cnt = R.status(p) != 0 ? 0 : R.children(p, buf);
                const Move want = Rules::real_move(p, moves[i]);
                bool found = false;
                for (int c = 0; c < cnt; ++c) found |= buf[c] == want;
                if (!found) throw fail(k, "move " + std::to_string(i - m0) + " is not legal here");
                p = R.moved(p, want);
                R.children(p, buf);
                h.push_back(p);
            }
            // older positions cannot repeat anything from here on (equal positions lie within `rev` plies)
            const size_t keep = std::min<size_t>({h.size(), static_cast<size_t>(p.rev) + 1u, hist_cap_for<Rules>()});
            h.erase(h.begin(), h.end() - static_cast<std::ptrdiff_t>(keep));
        } else {
            if (fen) throw fail(k, "a FEN is only accepted for chess (give the moves from the initial position)");
            p = R.initial();
            for (uint32_t i = m0; i < m1; ++i) {
                const uint32_t m = moves[i];
                if (R.status(p) != 0 || m >= static_cast<uint32_t>(R.moves_num()) || !(static_cast<uint32_t>(R.legal_mask(p) >> m) & 1u))
                    throw fail(k, "move " + std::to_string(i - m0) + " is not legal here");
                p = R.moved(p, static_cast<int>(m));
            }
            h.push_back(p);
        }
    }
    return out;
}

// The status of a history's last position as ChessGame reports it: a threefold repetition is a draw (chess/core.rs:441-449).
template <class Rules>
int analysis_root_status(const Rules& R, const std::vector<typename Rules::Pos>& h) {
    const auto& root = h.back();
    const int st = R.status(root);
    if (st != 0) return st;
    if constexpr (Rules::kChess) {
        int seen = 1;
        const int32_t H = static_cast<int32_t>(h.size());
        for (int32_t d = 2; d <= root.rev && d < H; d += 2)
            if (Rules::same(root, h[H - 1 - d])) ++seen;
        if (seen >= 3) return 3;
    }
    return 0;
}

template <class Rules, class Backend>
class AnalysisDriver {
    using Pos = typename Rules::Pos;
    using Move = typename Rules::Move;
    static constexpr bool kChess = Rules::kChess;

  public:
    // search_batch: the backend's (descents per minibatch; its result entries carry the minibatch counts when > 1)
    AnalysisDriver(const Rules& rules, const sp::Params& params, Backend& be, const std::vector<std::vector<Pos>>& histories,
                   std::vector<AnalysisResult>& out, uint32_t search_batch = 1)
        : R(rules), params_(params), be_(be), hist_(histories), out_(out), search_batch_(search_batch) {
        out_.assign(hist_.size(), AnalysisResult());
        job_of_slot_.assign(be.n_slots(), -1);
        cmd_stride_ = cmd_stride_for(be.max_children());
        result_stride_ = analysis_stride_for(be.max_children(), search_batch);
    }

    void run() {
        const uint32_t pops = be_.populations();
        for (uint32_t s = 0; s < be_.n_slots(); ++s) free_[be_.population_of(s)].push_back(s);
        std::deque<uint32_t> inflight;
        uint32_t wave = 0, next_pop = 0;
        const uint32_t depth = std::max<uint32_t>(1, be_.depth());
        for (;;) {
            bool submitted = false;
            uint32_t pop = next_pop;
            if (pops == 2 && !has_work(pop)) pop ^= 1u;
            if (has_work(pop)) {
                uint32_t n_roots = 0;
                const uint32_t n_cmds = fill(pop, wave, &n_roots);
                if (active_pop_[pop] > 0) {
                    uint32_t* hdr = reinterpret_cast<uint32_t*>(be_.cmd_block(wave));
                    hdr[0] = n_cmds;
                    hdr[1] = wave;
                    hdr[2] = hdr[3] = 0;
                    be_.submit(wave, pop, n_cmds, n_roots);
                    inflight.push_back(wave++);
                    submitted = true;
                    next_pop = pops == 2 ? (pop ^ 1u) : 0u;
                }
            }
            if (!inflight.empty() && (inflight.size() >= depth || !submitted)) {
                const uint32_t w = inflight.front();
                inflight.pop_front();
                uint32_t n_done = 0;
                const uint8_t* res = be_.wait(w, &n_done);
                for (uint32_t k = 0; k < n_done; ++k) on_result(res + static_cast<size_t>(k) * result_stride_);
            }
            if (active_ == 0 && inflight.empty() && next_ >= hist_.size()) break;
        }
        be_.read_counters(counters_);
    }

    // [0] simulations [1] evaluator rows [2] terminal leaves [3] cache hits, over the whole run
    const unsigned long long* counters() const { return counters_; }

  private:
    bool has_work(uint32_t pop) const { return active_pop_[pop] > 0 || (!free_[pop].empty() && next_ < hist_.size()); }

    // Commands for the population's next wave: the next positions go to its free slots while their histories fit the
    // wave's root block; positions whose game is already over are answered here without a search.
    uint32_t fill(uint32_t pop, uint32_t wave, uint32_t* n_roots) {
        uint8_t* block = be_.cmd_block(wave);
        Pos* roots = be_.roots_block(wave);
        const uint32_t cap = be_.roots_cap();
        uint32_t n_cmds = 0, staged = 0;
        while (!free_[pop].empty() && next_ < hist_.size()) {
            const std::vector<Pos>& h = hist_[next_];
            const int st = analysis_root_status(R, h);
            if (st != 0) {
                out_[next_++].status = static_cast<uint32_t>(st);
                continue;
            }
            const uint32_t len = static_cast<uint32_t>(h.size());
            if (staged + len > cap) break;  // the rest goes with a later wave
            const uint32_t slot = free_[pop].front();
            free_[pop].pop_front();
            std::copy(h.begin(), h.end(), roots + staged);
            Cmd c;
            std::memset(&c, 0, sizeof(c));
            c.slot = slot;
            c.flags = kCmdSetRoot;
            c.root_at = staged;
            c.root_len = len;
            uint8_t* at = block + 16 + static_cast<size_t>(n_cmds) * cmd_stride_;
            std::memset(at, 0, cmd_stride_);
            std::memcpy(at, &c, sizeof(c));
            staged += len;
            n_cmds += 1;
            job_of_slot_[slot] = static_cast<int64_t>(next_++);
            active_ += 1;
            active_pop_[pop] += 1;
        }
        *n_roots = staged;
        return n_cmds;
    }

    void on_result(const uint8_t* e) {
        const AnalysisHdr* ah = reinterpret_cast<const AnalysisHdr*>(e);
        const uint32_t slot = ah->slot, count = ah->count, pv_len = ah->pv_len;
        const uint32_t maxc = be_.max_children();
        if (slot >= job_of_slot_.size() || job_of_slot_[slot] < 0 || count > maxc || count == 0 || pv_len > kPvMax)
            throw sp::SpError{CATTUS_B200_EDEVICE, "device search posted a malformed result"};
        const size_t k = static_cast<size_t>(job_of_slot_[slot]);
        job_of_slot_[slot] = -1;
        read_analysis_entry(R, params_, hist_[k].back(), e, maxc, result_stride_, search_batch_, out_[k], probs_, weights_);
        const uint32_t pop = be_.population_of(slot);
        free_[pop].push_back(slot);
        active_ -= 1;
        active_pop_[pop] -= 1;
    }

    const Rules& R;
    sp::Params params_;
    Backend& be_;
    const std::vector<std::vector<Pos>>& hist_;
    std::vector<AnalysisResult>& out_;
    std::vector<int64_t> job_of_slot_;
    std::deque<uint32_t> free_[2];
    size_t next_ = 0;
    uint32_t active_ = 0, active_pop_[2] = {0, 0};
    uint32_t search_batch_ = 1, cmd_stride_ = 0, result_stride_ = 0;
    unsigned long long counters_[4] = {0, 0, 0, 0};
    std::vector<std::pair<Move, float>> probs_;
    std::vector<float> weights_;
};

// ---------------------------------------------------------------- accessors shared by the C ABI and the test emulation
inline int analysis_get(const std::vector<AnalysisResult>& r, uint32_t k, cattus_b200_analysis_position* out) {
    if (!out || k >= r.size()) return CATTUS_B200_ERANGE;
    if (out->struct_size != sizeof(cattus_b200_analysis_position)) return CATTUS_B200_EINVAL;
    const AnalysisResult& a = r[k];
    out->status = a.status;
    out->n_children = static_cast<uint32_t>(a.moves.size());
    out->pv_len = static_cast<uint32_t>(a.pv.size());
    out->simulations = a.simulations;
    out->best_move = a.best;
    out->pad = 0;
    out->q = a.q;
    return CATTUS_B200_OK;
}

inline int analysis_children(const std::vector<AnalysisResult>& r, uint32_t k, uint16_t* moves, uint32_t* visits, float* w, float* priors, uint32_t cap) {
    if (k >= r.size()) return CATTUS_B200_ERANGE;
    const AnalysisResult& a = r[k];
    const size_t n = a.moves.size();
    if (cap < n) return CATTUS_B200_ERANGE;
    for (size_t i = 0; i < n; ++i) {
        if (moves) moves[i] = a.moves[i];
        if (visits) visits[i] = a.visits[i];
        if (w) w[i] = a.w[i];
        if (priors) priors[i] = a.prior[i];
    }
    return CATTUS_B200_OK;
}

inline int analysis_batches(const std::vector<AnalysisResult>& r, uint32_t k, uint32_t* minibatches, uint32_t* collisions) {
    if (k >= r.size()) return CATTUS_B200_ERANGE;
    if (minibatches) *minibatches = r[k].minibatches;
    if (collisions) *collisions = r[k].collisions;
    return CATTUS_B200_OK;
}

inline int analysis_pv(const std::vector<AnalysisResult>& r, uint32_t k, uint16_t* pv, uint32_t cap) {
    if (k >= r.size() || !pv) return CATTUS_B200_ERANGE;
    const AnalysisResult& a = r[k];
    if (cap < a.pv.size()) return CATTUS_B200_ERANGE;
    for (size_t i = 0; i < a.pv.size(); ++i) pv[i] = a.pv[i];
    return CATTUS_B200_OK;
}

}  // namespace ds
