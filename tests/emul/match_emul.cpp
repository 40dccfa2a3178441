// TEST INFRASTRUCTURE -- never part of the product library.
//
// Match play from openings (cattus_b200/csrc/dsearch_match.hpp) over the host emulation of the device-resident search
// (dsearch_emul.cpp, included whole: its EmulBackend gains the root upload here and keeps the self-play result layout),
// with two callback evaluators.  The CPU tests compare it with the emulated self-play driver and with oracle/mcts.py's
// play_game from the same starting history.
#include "dsearch_emul.cpp"

#include "../../cattus_b200/csrc/dsearch_match.hpp"

namespace {

template <class Rules>
struct EmulMatchBackend : EmulBackend<Rules> {
    using Base = EmulBackend<Rules>;
    using Pos = typename Rules::Pos;
    std::vector<Pos> roots;

    EmulMatchBackend(const Rules& rules, const void* blob, uint32_t n_slots, uint32_t pool_words, uint32_t depth, const sp::Params params[2],
                     cattus_b200_eval_fn f1, cattus_b200_eval_fn f2, uint32_t cache_size, uint32_t roots_cap)
        : Base(rules, blob, n_slots, pool_words, depth, params, f1, nullptr, f2, nullptr, cache_size) {
        roots.assign(roots_cap, Pos());
        this->p.roots = roots.data();
        this->p2.roots = roots.data();
    }
    Pos* roots_block(uint32_t) { return roots.data(); }
    uint32_t roots_cap() const { return static_cast<uint32_t>(roots.size()); }
    void submit(uint32_t wave, uint32_t pop, uint32_t n_cmds, uint32_t) { Base::submit(wave, pop, n_cmds); }
};

struct MatchEmulResult {
    ds::MatchResult res;
    std::string error;
};

template <class Rules>
void match_emul(const Rules& rules, const void* blob, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_match_side* side_b, uint32_t n,
                const char* const* fens, const uint16_t* moves, const uint32_t* offsets, uint32_t n_slots, uint32_t pool_words, uint32_t depth,
                uint32_t roots_cap, cattus_b200_eval_fn fa, cattus_b200_eval_fn fb, ds::MatchResult& out) {
    sp::Params params[2];
    ds::match_params(*cfg, side_b, params);
    const auto openings = ds::match_openings(rules, n, fens, moves, offsets, out.opening_status);
    const uint32_t games = ds::match_games(out.opening_status);
    if (!games) return;
    EmulMatchBackend<Rules> be(rules, blob, std::min(n_slots, games), pool_words, depth, params, fa, fb, cfg->cache_size,
                               std::max(roots_cap, ds::hist_cap_for<Rules>()));
    ds::match_play(rules, *cfg, params, be, openings, out);
}

}  // namespace

extern "C" {

// fb NULL: one evaluator for both sides.  depth: the test knobs of dsearch_emul_run; roots_cap: history positions one wave
// can upload (raised to the ring size)
void* match_emul_run(cattus_b200_eval_fn fa, cattus_b200_eval_fn fb, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_match_side* side_b,
                     uint32_t n, const char* const* fens, const uint16_t* moves, const uint32_t* offsets, uint32_t n_slots, uint32_t pool_words,
                     uint32_t depth, uint32_t roots_cap) {
    std::unique_ptr<MatchEmulResult> r(new MatchEmulResult());
    try {
        if (cfg->game == CATTUS_B200_GAME_HEX) {
            if (cfg->board_size <= 8) {
                sp::HexRulesT<uint64_t> rules(static_cast<int>(cfg->board_size));
                match_emul(rules, &rules, cfg, side_b, n, fens, moves, offsets, n_slots, pool_words, depth, roots_cap, fa, fb, r->res);
            } else {
                sp::HexRulesT<sp::u128> rules(static_cast<int>(cfg->board_size));
                match_emul(rules, &rules, cfg, side_b, n, fens, moves, offsets, n_slots, pool_words, depth, roots_cap, fa, fb, r->res);
            }
        } else if (cfg->game == CATTUS_B200_GAME_CHESS) {
            sp::ChessRules rules;
            match_emul(rules, &sp::chess_tables(), cfg, side_b, n, fens, moves, offsets, n_slots, pool_words, depth, roots_cap, fa, fb, r->res);
        } else {
            sp::TttRules rules;
            match_emul(rules, &rules, cfg, side_b, n, fens, moves, offsets, n_slots, pool_words, depth, roots_cap, fa, fb, r->res);
        }
    } catch (const sp::SpError& e) {
        r->error = e.msg.empty() ? "error" : e.msg;
    }
    return r.release();
}
const char* match_emul_error(void* h) { return static_cast<MatchEmulResult*>(h)->error.c_str(); }
int match_emul_summary(const void* h, cattus_b200_match_summary* out) { return ds::match_summary(static_cast<const MatchEmulResult*>(h)->res, out); }
int match_emul_opening_status(const void* h, uint32_t k, uint32_t* st) {
    return ds::match_opening_status(static_cast<const MatchEmulResult*>(h)->res, k, st);
}
int match_emul_game(const void* h, uint32_t k, cattus_b200_match_game* out) { return ds::match_game(static_cast<const MatchEmulResult*>(h)->res, k, out); }
int match_emul_game_moves(const void* h, uint32_t k, uint16_t* moves, uint32_t cap) {
    return ds::match_game_moves(static_cast<const MatchEmulResult*>(h)->res, k, moves, cap);
}
void match_emul_free(void* h) { delete static_cast<MatchEmulResult*>(h); }
}
