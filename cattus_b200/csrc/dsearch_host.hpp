// Host half of the device-resident self-play (dsearch_core.hpp holds the per-simulation half that runs on the GPU).
//
// What happens here is what the reference does ONCE PER MOVE (training/self-play/src/self_play.rs:179-246,
// engine/src/mcts/mod.rs:364-446): turn the finished search's root visit counts into move probabilities, choose the move
// (temperature policy, the game's random stream), advance the game, decide whether it is over, write the .traindata
// entries, and draw the Dirichlet sample for the next search's root.  Each wave of the device pipeline posts the
// searches that just finished; this driver answers with one command per game (new game / move + who searches + the
// noise sample) that the device applies at the start of a later wave.  Several waves are kept in flight so the GPU never
// waits for the host.
//
// `Backend` is the transport: the CUDA one (dsearch.cuh) launches the captured wave graph and reads results from mapped
// pinned memory; the one in tests/emul runs the same per-slot code on the host for the CPU parity tests.
//
// With an opening source (a match between two networks, dsearch_match.hpp) game 2k + c starts from opening k instead of
// the initial position: a kCmdSetRoot command installs the opening with its history, which the backend uploads with the
// wave (roots_block / roots_cap).  Everything else is the self-play game loop.
//
// With minibatches (a side's search_batch > 1, DESIGN.md section 16) the backend runs the minibatch kernels, and each
// finished search posts its minibatch and collision counts in ResultHdr::pad; the driver sums them per side.
#pragma once

#include <deque>
#include <type_traits>
#include <utility>
#include <vector>

#include "dsearch_core.hpp"
#include "sp_common.hpp"

namespace ds {

inline uint32_t cmd_stride_for(uint32_t max_children) { return (static_cast<uint32_t>(sizeof(Cmd)) + 4u * max_children + 15u) & ~15u; }
inline uint32_t result_stride_for(uint32_t max_children) { return (static_cast<uint32_t>(sizeof(ResultHdr)) + 6u * max_children + 15u) & ~15u; }

// whether a backend can upload root histories with a wave (kCmdSetRoot)
template <class B, class = void>
struct HasRootUpload : std::false_type {};
template <class B>
struct HasRootUpload<B, std::void_t<decltype(std::declval<B&>().roots_block(0u))>> : std::true_type {};

template <class Rules, class Backend>
class Driver {
    using Pos = typename Rules::Pos;
    using Move = typename Rules::Move;
    static constexpr bool kChess = Rules::kChess;

    struct Game {
        bool active = false;
        uint32_t game_idx = 0;
        sp::SplitMix64 rng;
        std::vector<Pos> history;
        size_t hist_base = 0;  // positions of `history` before the game's first position (an opening's history)
        int cur = 0;
        sp::GameRecord rec;
        std::vector<std::pair<Pos, std::vector<std::pair<Move, float>>>> pending_entries;
        bool repetition = false;  // ChessGame::repetition_detected (chess/core.rs:441-449)
        bool has_last_root[2] = {false, false};
        Pos last_root[2];  // the position each player searched last: searching it again keeps the tree and adds no noise
        sp::Clock::time_point search_t0;
    };

  public:
    // openings (optional): per opening k, the history kCmdSetRoot loads (oldest first, the opening's position last; at most
    // the backend's history ring); games 2k and 2k + 1 start there.  An empty history: the opening is not played.
    // cfg.games_num must be twice the number of openings.  Such games keep records (moves, winner, termination) but write
    // no training data.  search_batch (optional): the backend's descents per minibatch of model 1's and model 2's searches.
    Driver(const Rules& rules, const cattus_b200_selfplay_cfg& cfg, const sp::Params params[2], Backend& be, sp::Shared& sh,
           const std::vector<std::vector<Pos>>* openings = nullptr, const uint32_t* search_batch = nullptr)
        : R(rules), cfg_(cfg), be_(be), sh_(sh), openings_(openings), batched_(search_batch && (search_batch[0] > 1 || search_batch[1] > 1)) {
        params_[0] = params[0];
        params_[1] = params[1];
        games_.resize(be.n_slots());
        cmd_stride_ = cmd_stride_for(be.max_children());
        result_stride_ = result_stride_for(be.max_children());
    }

    void run() {
        // Two POPULATIONS of slots (when the backend has two evaluator lanes) take waves in turn, each on its own stream: while
        // one population's leaves are in the evaluator, the other's select / expand kernels run beside it, and a slot that
        // finished a search gets its command in the very next wave of its population.
        const uint32_t n = be_.n_slots();
        for (uint32_t s = 0; s < n; ++s) start_next_game(s);
        std::deque<uint32_t> inflight;
        uint32_t wave = 0, next_pop = 0;
        const uint32_t depth = std::max<uint32_t>(1, be_.depth());
        const uint32_t pops = be_.populations();
        for (;;) {
            bool submitted = false;
            const auto ta = sp::Clock::now();
            uint32_t pop = next_pop;
            if (pops == 2 && active_pop_[pop] == 0 && cmds_[pop].empty()) pop ^= 1u;  // nothing to do there: give the turn away
            if (active_pop_[pop] > 0 || !cmds_[pop].empty()) {
                uint8_t* block = be_.cmd_block(wave);
                uint32_t n_cmds = static_cast<uint32_t>(cmds_[pop].size() / cmd_stride_);
                uint32_t* hdr = reinterpret_cast<uint32_t*>(block);
                if (n_cmds) std::memcpy(block + 16, cmds_[pop].data(), cmds_[pop].size());
                cmds_[pop].clear();
                uint32_t n_roots = 0;
                if constexpr (HasRootUpload<Backend>::value)
                    n_cmds += stage_roots(pop, wave, block + 16 + static_cast<size_t>(n_cmds) * cmd_stride_, &n_roots);
                hdr[0] = n_cmds;
                hdr[1] = wave;
                hdr[2] = hdr[3] = 0;
                if constexpr (HasRootUpload<Backend>::value)
                    be_.submit(wave, pop, n_cmds, n_roots);
                else
                    be_.submit(wave, pop, n_cmds);
                inflight.push_back(wave++);
                submitted = true;
                waves_ += 1;
                next_pop = pops == 2 ? (pop ^ 1u) : 0u;
            }
            const auto tb = sp::Clock::now();
            if (!inflight.empty() && (inflight.size() >= depth || !submitted)) {
                const uint32_t w = inflight.front();
                inflight.pop_front();
                uint32_t n_done = 0;
                const uint8_t* res = be_.wait(w, &n_done);
                const auto tc = sp::Clock::now();
                for (uint32_t k = 0; k < n_done; ++k) on_result(res + static_cast<size_t>(k) * result_stride_);
                t_wait_ += std::chrono::duration<double>(tc - tb).count();
                t_process_ += std::chrono::duration<double>(sp::Clock::now() - tc).count();
            }
            t_submit_ += std::chrono::duration<double>(tb - ta).count();
            if (active_ == 0 && inflight.empty()) break;
        }
        unsigned long long c[4] = {0, 0, 0, 0};
        be_.read_counters(c);
        if (std::getenv("CATTUS_B200_DSEARCH_PROFILE"))  // where the host thread's time went: a large `wait` share means the GPU is the limit
            std::fprintf(stderr, "device search host thread: %llu waves, submit %.3f s, wait (GPU) %.3f s, per-move work %.3f s (%llu searches)\n",
                         static_cast<unsigned long long>(waves_), t_submit_, t_wait_, t_process_, static_cast<unsigned long long>(searches_));
        std::lock_guard<std::mutex> g(sh_.mu);
        sh_.simulations += c[0];
        sh_.evaluations += c[1];
        sh_.cache_misses += c[1];  // every evaluator row was a miss of the device-side cache (or there is no cache)
        sh_.cache_hits += c[3];
        sh_.terminal += c[2];
        sh_.batches += waves_;
        sh_.searches += searches_;
        sh_.w1 += w1_;
        sh_.w2 += w2_;
        sh_.d += d_;
        sh_.games += games_done_;
        for (int s = 0; s < 2; ++s) {
            sh_.minibatches[s] += minibatches_[s];
            sh_.collisions[s] += collisions_[s];
        }
        sh_.search_duration = search_duration_;
    }

  private:
    // self_play.rs:183-205: the next game index of this partition, a fresh game, the first search's command
    void start_next_game(uint32_t slot) {
        Game& g = games_[slot];
        const uint32_t stride = std::max<uint32_t>(1, cfg_.game_stride);
        uint64_t idx;
        do {
            const uint32_t k = sh_.next_game.fetch_add(1);
            idx = static_cast<uint64_t>(cfg_.first_game) + static_cast<uint64_t>(k) * stride;
            if (idx >= cfg_.games_num) {
                g.active = false;
                return;
            }
        } while (openings_ && (*openings_)[idx / 2].empty());
        g = Game();
        g.active = true;
        g.game_idx = static_cast<uint32_t>(idx);
        g.rng = sp::SplitMix64(sp::game_seed(cfg_.seed, g.game_idx));
        g.rec.game_idx = g.game_idx;
        active_ += 1;
        active_pop_[be_.population_of(slot)] += 1;
        if (openings_) {
            const std::vector<Pos>& h = (*openings_)[idx / 2];
            g.history = h;
            g.hist_base = h.size() - 1;
            begin_move(slot, kCmdSetRoot, 0);
        } else {
            g.history.push_back(R.initial());
            begin_move(slot, kCmdNewGame, 0);
        }
    }

    // Moves the population's waiting kCmdSetRoot commands into the wave's command block at `at` while their histories fit
    // the wave's root block; the rest wait for a later wave (their slots stay idle on the device until then).
    uint32_t stage_roots(uint32_t pop, uint32_t wave, uint8_t* at, uint32_t* n_roots) {
        std::vector<uint8_t>& wait = set_root_[pop];
        Pos* roots = be_.roots_block(wave);
        const uint32_t cap = be_.roots_cap();
        uint32_t staged = 0, n = 0;
        size_t off = 0;
        for (; off < wait.size(); off += cmd_stride_, ++n) {
            Cmd c;
            std::memcpy(&c, wait.data() + off, sizeof(c));
            const std::vector<Pos>& h = games_[c.slot].history;
            const uint32_t len = static_cast<uint32_t>(h.size());
            if (staged + len > cap) break;
            std::copy(h.begin(), h.end(), roots + staged);
            c.root_at = staged;
            c.root_len = len;
            std::memcpy(at + off, wait.data() + off, cmd_stride_);
            std::memcpy(at + off, &c, sizeof(c));
            staged += len;
        }
        wait.erase(wait.begin(), wait.begin() + static_cast<std::ptrdiff_t>(off));
        *n_roots = staged;
        return n;
    }

    // One step of the game loop at a position that is about to be searched (or ends the game).
    void begin_move(uint32_t slot, uint32_t flags, uint32_t move) {
        Game& g = games_[slot];
        Pos& pos = g.history.back();
        int n_legal;
        if constexpr (kChess) {
            Move buf[256];
            n_legal = R.children(pos, buf);  // settles status()
        } else {
            n_legal = R.status(pos) != 0 ? 0 : sp::popcount128(R.legal_mask(pos));
        }
        int st = g.repetition ? 3 : R.status(pos);  // ChessGame::status: a threefold repetition is a draw
        g.rec.termination = g.repetition ? sp::kEndRepetition : sp::kEndRules;
        if (st == 0 && cfg_.max_moves && g.rec.moves.size() >= cfg_.max_moves) {  // bounded runs only (not in the reference)
            st = 3;
            g.rec.termination = sp::kEndMaxMoves;
        }
        if (st != 0) {
            finish_game(g, st);
            active_ -= 1;
            active_pop_[be_.population_of(slot)] -= 1;
            start_next_game(slot);
            return;
        }
        int who = pos.turn;  // self_play.rs:198-205
        if (g.game_idx % 2 == 1) who = 3 - who;
        g.cur = who - 1;
        const sp::Params& P = params_[g.cur];
        // add_dirichlet_noise (mod.rs:419-446) runs once per search, on the root, as soon as the root has children: at
        // tree reuse or when the first simulation expands it -- unless the very same position is searched again
        // (remove_all_but_subtree returns early, mod.rs:304-306)
        uint32_t noise_n = 0;
        const bool same_root = g.has_last_root[g.cur] && R.same(g.last_root[g.cur], pos);
        if (P.noise_alpha != 0.0f && P.noise_eps != 0.0f && n_legal >= 2 && !same_root) {
            const double tot = sp::draw_noise(g.rng, P.noise_alpha, n_legal, noise_);
            noise_n = static_cast<uint32_t>(n_legal);
            nz_.resize(noise_n);
            for (uint32_t i = 0; i < noise_n; ++i) nz_[i] = static_cast<float>(noise_[i] / tot);
        }
        g.search_t0 = sp::Clock::now();
        // kCmdSetRoot waits in its own queue: its history goes with whichever wave has room for it (stage_roots)
        std::vector<uint8_t>& cmds = (flags == kCmdSetRoot ? set_root_ : cmds_)[be_.population_of(slot)];
        const size_t at = cmds.size();
        cmds.resize(at + cmd_stride_, 0);
        Cmd c;
        std::memset(&c, 0, sizeof(c));
        c.slot = slot;
        c.flags = flags;
        c.move = move;
        c.cur = static_cast<uint32_t>(g.cur);
        c.noise_n = noise_n;
        std::memcpy(cmds.data() + at, &c, sizeof(c));
        if (noise_n) std::memcpy(cmds.data() + at + sizeof(Cmd), nz_.data(), sizeof(float) * noise_n);
    }

    // the rest of calc_moves_probabilities + choose_move_from_probabilities + the game step (mod.rs:364-417,
    // self_play.rs:207-217)
    void on_result(const uint8_t* e) {
        const ResultHdr* rh = reinterpret_cast<const ResultHdr*>(e);
        const uint32_t slot = rh->slot, count = rh->count;
        if (slot >= games_.size() || !games_[slot].active || count > be_.max_children())
            throw sp::SpError{CATTUS_B200_EDEVICE, "device search posted a malformed result"};
        Game& g = games_[slot];
        const uint32_t* rn = reinterpret_cast<const uint32_t*>(e + sizeof(ResultHdr));
        const uint16_t* rm = reinterpret_cast<const uint16_t*>(e + sizeof(ResultHdr) + 4u * be_.max_children());
        const sp::Params& P = params_[g.cur];
        // the one-leaf kernels run a search as sim_num rounds of one descent each and post no counts
        minibatches_[g.cur] += batched_ ? rh->pad[0] : P.sim_num;
        collisions_[g.cur] += batched_ ? rh->pad[1] : 0u;
        std::vector<std::pair<Move, float>> probs;
        probs.reserve(count);
        uint32_t total = 0;
        for (uint32_t i = 0; i < count; ++i) total += rn[i];
        for (int32_t i = static_cast<int32_t>(count) - 1; i >= 0; --i)  // edges() order
            probs.emplace_back(static_cast<Move>(rm[i]), static_cast<float>(rn[i]) / static_cast<float>(total));
        const double secs = std::chrono::duration<double>(sp::Clock::now() - g.search_t0).count();
        search_duration_ = (1.0 - 0.99) * search_duration_ + 0.99 * secs;  // RunningAverage(0.99), util/metric.rs:1-20
        searches_ += 1;
        if (probs.empty()) throw sp::SpError{CATTUS_B200_EINVAL, "search produced no moves"};
        // the temperature policy counts moves from the game's first position (an opening's history does not count)
        const int chosen = sp::choose_move(P, g.history.size() - g.hist_base, probs, g.rng, weights_);
        const Move mv = probs[chosen].first;
        g.last_root[g.cur] = g.history.back();
        g.has_last_root[g.cur] = true;
        g.pending_entries.emplace_back(g.history.back(), std::move(probs));
        if constexpr (kChess) {
            g.rec.moves.push_back(Rules::real_move(g.history.back(), mv));
            Pos np = R.moved(g.history.back(), mv);
            Move buf[256];
            R.children(np, buf);  // settles status()
            // ChessGame::play_single_turn (chess/core.rs:441-449): the third occurrence of a position ends the game
            int seen = 1;
            const int32_t H = static_cast<int32_t>(g.history.size());
            for (int32_t d = 2; d <= np.rev && d <= H; d += 2)
                if (Rules::same(np, g.history[H - d])) ++seen;
            if (seen >= 3) g.repetition = true;
            g.history.push_back(np);
        } else {
            g.rec.moves.push_back(mv);
            g.history.push_back(R.moved(g.history.back(), mv));
        }
        begin_move(slot, kCmdMove, static_cast<uint32_t>(mv));
    }

    void finish_game(Game& g, int status) {
        const uint8_t winner = status == 3 ? 0 : static_cast<uint8_t>(status);
        g.rec.winner = winner;
        for (size_t pos_idx = 0; !openings_ && pos_idx < g.pending_entries.size(); ++pos_idx) {
            auto& pe = g.pending_entries[pos_idx];
            std::vector<uint8_t> bytes;
            const int dir = sp::make_entry(R, g.game_idx, pe.first, pe.second, winner, bytes);
            if (cfg_.out_dir1 && cfg_.out_dir2) sp::write_entry_file(dir == 1 ? cfg_.out_dir1 : cfg_.out_dir2, g.game_idx, pos_idx, bytes);
            if (cfg_.keep_records) {
                g.rec.entries.push_back(std::move(bytes));
                g.rec.entry_dir.push_back(static_cast<uint8_t>(dir));
            }
        }
        // winner counters: self_play.rs:226-241
        uint8_t credited = winner;
        if (credited && g.game_idx % 2 == 1) credited = static_cast<uint8_t>(3 - credited);
        if (credited == 0)
            d_ += 1;
        else if (credited == 1)
            w1_ += 1;
        else
            w2_ += 1;
        games_done_ += 1;
        if (cfg_.keep_records || openings_) {
            std::lock_guard<std::mutex> lk(sh_.mu);
            sh_.records.push_back(std::move(g.rec));
        }
        g.pending_entries.clear();
    }

    const Rules& R;
    const cattus_b200_selfplay_cfg& cfg_;
    Backend& be_;
    sp::Shared& sh_;
    sp::Params params_[2];
    const std::vector<std::vector<Pos>>* openings_;
    const bool batched_;
    std::vector<Game> games_;
    std::vector<uint8_t> cmds_[2];      // commands for each population's next wave
    std::vector<uint8_t> set_root_[2];  // kCmdSetRoot commands waiting for room in a wave's root block
    uint32_t cmd_stride_ = 0, result_stride_ = 0;
    uint32_t active_ = 0, active_pop_[2] = {0, 0};
    uint64_t waves_ = 0, searches_ = 0, minibatches_[2] = {0, 0}, collisions_[2] = {0, 0};
    uint32_t w1_ = 0, w2_ = 0, d_ = 0, games_done_ = 0;
    double search_duration_ = 0.0, t_submit_ = 0.0, t_wait_ = 0.0, t_process_ = 0.0;
    std::vector<double> noise_;
    std::vector<float> nz_, weights_;
};

}  // namespace ds
