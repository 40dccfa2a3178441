// Host half of match play between two networks from an opening suite (include/cattus_b200_match.h) on the
// device-resident search.
//
// A match is self-play with an opening source: ds::Driver (dsearch_host.hpp) plays game 2k + c from opening k, model 1
// (A) as player 1 in even games, with the self-play game loop unchanged.  This file turns the C ABI's inputs into that
// driver's: each opening's history (analysis_histories, the same checks and the same history kCmdSetRoot loads for an
// analysis), the two sides' MctsParams, the driver's config; and reads the games back.  `Backend` is the self-play
// transport with the root upload (dsearch.cuh's DsCudaBackend built with a roots_cap, tests/emul's emulation).
#pragma once

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/cattus_b200_match.h"
#include "dsearch_analysis.hpp"
#include "dsearch_host.hpp"
#include "sp_common.hpp"

namespace ds {

struct MatchResult {
    std::vector<uint32_t> opening_status;  // per opening: 0 played; otherwise the finished position's status, not played
    std::vector<sp::GameRecord> games;     // by game index 2k + c
    uint32_t a_wins = 0, b_wins = 0, draws = 0;
    uint64_t simulations = 0, evaluations = 0;
    uint64_t minibatches[2] = {0, 0}, collisions[2] = {0, 0};  // per side (A, B)
    double seconds = 0.0;
};

// Each side's descents per minibatch from the C ABI's options: NULL, or 0 or 1 for a side, is one leaf in flight.
inline void match_search_batch(const cattus_b200_match_opts* opts, uint32_t out[2]) {
    out[0] = out[1] = 1;
    if (!opts) return;
    if (opts->struct_size != sizeof(cattus_b200_match_opts)) throw sp::SpError{CATTUS_B200_EINVAL, "match opts struct_size mismatch"};
    out[0] = opts->search_batch_a ? opts->search_batch_a : 1u;
    out[1] = opts->search_batch_b ? opts->search_batch_b : 1u;
}

// The two sides' MctsParams: cfg's, with side B's sim_num / explore_factor where side_b gives them.
inline void match_params(const cattus_b200_selfplay_cfg& cfg, const cattus_b200_match_side* side_b, sp::Params out[2]) {
    if (cfg.struct_size != sizeof(cattus_b200_selfplay_cfg)) throw sp::SpError{CATTUS_B200_EINVAL, "selfplay cfg struct_size mismatch"};
    if (cfg.game == CATTUS_B200_GAME_HEX) {
        if (cfg.board_size < 2 || cfg.board_size > 11) throw sp::SpError{CATTUS_B200_EINVAL, "hex board_size must be 2..11"};
    } else if (cfg.game != CATTUS_B200_GAME_TTT && cfg.game != CATTUS_B200_GAME_CHESS) {
        throw sp::SpError{CATTUS_B200_EINVAL, "unknown game"};
    }
    out[0] = sp::parse_params(&cfg);
    out[1] = out[0];
    if (!side_b) return;
    if (side_b->struct_size != sizeof(cattus_b200_match_side)) throw sp::SpError{CATTUS_B200_EINVAL, "match side struct_size mismatch"};
    if (side_b->sim_num) {
        if (side_b->sim_num < 2) throw sp::SpError{CATTUS_B200_EINVAL, "match: side B's sim_num must be > 1 (mcts/mod.rs:157)"};
        out[1].sim_num = side_b->sim_num;
    }
    if (side_b->explore_factor >= 0.0f)
        out[1].explore_factor = side_b->explore_factor;
    else if (!(side_b->explore_factor < 0.0f))
        throw sp::SpError{CATTUS_B200_EINVAL, "match: side B's explore_factor is NaN"};
}

// The driver's config: 2n games from game index 0, records kept, no training data.
inline cattus_b200_selfplay_cfg match_cfg(const cattus_b200_selfplay_cfg& cfg, uint32_t n) {
    cattus_b200_selfplay_cfg c = cfg;
    c.games_num = 2u * n;
    c.first_game = 0;
    c.game_stride = 1;
    c.out_dir1 = c.out_dir2 = nullptr;
    c.keep_records = 1;
    return c;
}

// Each opening's history as kCmdSetRoot loads it; an opening whose position is already finished gets its status in
// `status` and an empty history (the driver does not play it).
template <class Rules>
std::vector<std::vector<typename Rules::Pos>> match_openings(const Rules& R, uint32_t n, const char* const* fens, const uint16_t* moves,
                                                             const uint32_t* move_offsets, std::vector<uint32_t>& status) {
    if (n > 0x7FFFFFFFu) throw sp::SpError{CATTUS_B200_ERANGE, "match: too many openings"};
    auto hist = analysis_histories(R, n, fens, moves, move_offsets, "opening");
    status.assign(n, 0u);
    for (uint32_t k = 0; k < n; ++k) {
        const int st = analysis_root_status(R, hist[k]);
        if (st != 0) {
            status[k] = static_cast<uint32_t>(st);
            hist[k].clear();
        }
    }
    return hist;
}

// Plays the openings' games on `be` (its slots: at most the number of games) and fills out's games and counts.
template <class Rules, class Backend>
void match_play(const Rules& R, const cattus_b200_selfplay_cfg& cfg, const sp::Params params[2], Backend& be,
                const std::vector<std::vector<typename Rules::Pos>>& openings, MatchResult& out, const uint32_t* search_batch = nullptr) {
    const cattus_b200_selfplay_cfg mc = match_cfg(cfg, static_cast<uint32_t>(openings.size()));
    sp::Shared sh;
    Driver<Rules, Backend> drv(R, mc, params, be, sh, &openings, search_batch);
    drv.run();
    out.games = std::move(sh.records);
    std::sort(out.games.begin(), out.games.end(), [](const sp::GameRecord& a, const sp::GameRecord& b) { return a.game_idx < b.game_idx; });
    out.a_wins = sh.w1;  // the driver credits wins to model 1 / model 2 whatever colour they played
    out.b_wins = sh.w2;
    out.draws = sh.d;
    out.simulations = sh.simulations;
    out.evaluations = sh.evaluations;
    for (int s = 0; s < 2; ++s) {
        out.minibatches[s] = sh.minibatches[s];
        out.collisions[s] = sh.collisions[s];
    }
}

// The games a match needs slots for: two per opening that is played.
inline uint32_t match_games(const std::vector<uint32_t>& status) {
    uint32_t g = 0;
    for (uint32_t st : status) g += st == 0 ? 2u : 0u;
    return g;
}

// ---------------------------------------------------------------- accessors shared by the C ABI and the test emulation
inline int match_summary(const MatchResult& r, cattus_b200_match_summary* out) {
    if (!out) return CATTUS_B200_EINVAL;
    if (out->struct_size != sizeof(cattus_b200_match_summary)) return CATTUS_B200_EINVAL;
    out->a_wins = r.a_wins;
    out->b_wins = r.b_wins;
    out->draws = r.draws;
    out->games = static_cast<uint32_t>(r.games.size());
    out->openings = static_cast<uint32_t>(r.opening_status.size());
    out->skipped = 0;
    for (uint32_t st : r.opening_status) out->skipped += st != 0 ? 1u : 0u;
    for (uint32_t& p : out->pairs) p = 0;
    // A's half points in each game, summed over the opening's two games (both are always played)
    for (size_t i = 0; i + 1 < r.games.size(); i += 2) {
        uint32_t halves = 0;
        for (size_t j = i; j < i + 2; ++j) {
            const sp::GameRecord& g = r.games[j];
            const uint32_t a_player = g.game_idx % 2 == 0 ? 1u : 2u;
            halves += g.winner == 0 ? 1u : (g.winner == a_player ? 2u : 0u);
        }
        out->pairs[halves] += 1;
    }
    out->simulations = r.simulations;
    out->evaluations = r.evaluations;
    out->seconds = r.seconds;
    return CATTUS_B200_OK;
}

inline int match_opening_status(const MatchResult& r, uint32_t k, uint32_t* status) {
    if (!status) return CATTUS_B200_EINVAL;
    if (k >= r.opening_status.size()) return CATTUS_B200_ERANGE;
    *status = r.opening_status[k];
    return CATTUS_B200_OK;
}

inline int match_game(const MatchResult& r, uint32_t k, cattus_b200_match_game* out) {
    if (!out) return CATTUS_B200_EINVAL;
    if (k >= r.games.size()) return CATTUS_B200_ERANGE;
    if (out->struct_size != sizeof(cattus_b200_match_game)) return CATTUS_B200_EINVAL;
    const sp::GameRecord& g = r.games[k];
    out->opening = g.game_idx / 2;
    out->a_is_player1 = g.game_idx % 2 == 0 ? 1u : 0u;
    out->winner = g.winner;
    out->termination = g.termination;
    out->n_moves = static_cast<uint32_t>(g.moves.size());
    return CATTUS_B200_OK;
}

inline int match_batches(const MatchResult& r, uint32_t side, uint64_t* minibatches, uint64_t* collisions) {
    if (side > 1) return CATTUS_B200_ERANGE;
    if (minibatches) *minibatches = r.minibatches[side];
    if (collisions) *collisions = r.collisions[side];
    return CATTUS_B200_OK;
}

inline int match_game_moves(const MatchResult& r, uint32_t k, uint16_t* moves, uint32_t cap) {
    if (k >= r.games.size() || !moves) return CATTUS_B200_ERANGE;
    const auto& m = r.games[k].moves;
    if (cap < m.size()) return CATTUS_B200_ERANGE;
    std::copy(m.begin(), m.end(), moves);
    return CATTUS_B200_OK;
}

}  // namespace ds
