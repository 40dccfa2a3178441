/* cattus_b200_analysis.h -- C ABI of the batched MCTS analysis of given positions.
 *
 * Every position is searched on the device-resident search of cattus_b200_selfplay_run's `device_games` mode (search
 * trees in HBM, one warp per tree), thousands at a time, as a fresh MctsPlayer (engine/src/mcts/mod.rs:335-385) with no
 * root noise searches it: the same visit counts, the same best move as cattus_b200_chess_search_go with noise off and
 * temperature 0.  A result depends on the position, its history, the network and the mcts.* fields alone -- not on
 * device_games, device_waves_in_flight, the cache or where the position falls in the input.
 */
#ifndef CATTUS_B200_ANALYSIS_H
#define CATTUS_B200_ANALYSIS_H

#include <stddef.h>
#include <stdint.h>

#include "cattus_b200.h"
#include "cattus_b200_selfplay.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cattus_b200_analysis cattus_b200_analysis_t;

typedef struct cattus_b200_analysis_position {
    uint32_t struct_size;
    uint32_t status;      /* 0: searched.  1 / 2: the game is over and that player won; 3: draw (threefold repetition of the
                           * given history included).  A finished position is not searched and has no children. */
    uint32_t n_children;  /* legal moves of the position (searched positions) */
    uint32_t pv_len;      /* plies of the principal variation, <= 16 */
    uint32_t simulations; /* develop_tree iterations of the search (cfg->sim_num) */
    uint16_t best_move;   /* choose_move_from_probabilities at temperature 0 over the visit distribution */
    uint16_t pad;
    float q;              /* sum W / sum N over the root's children: the side to move's mean score, in [-1, 1] */
} cattus_b200_analysis_position;

/* Searches n positions with `model` (any precision of the handle, FP8 included).  Position k is fens[k] followed by
 * moves[move_offsets[k] .. move_offsets[k + 1]).
 *   fens:          chess FENs (board, side, castling, en passant; clocks are ignored); NULL or fens[k] NULL = the game's
 *                  initial position.  Hex and tic-tac-toe take no FEN: fens[k] must be NULL.
 *   moves:         each game's move encoding -- chess from | to << 6 | promotion << 12 in real board coordinates
 *                  (include/cattus_b200_chess.h), hex and tic-tac-toe cell index row * S + col.
 *   move_offsets:  n + 1 ascending entries; NULL = no moves.
 * cfg: game / board_size, mcts.* (sim_num, explore_factor; prior_noise_epsilon must be 0), cache_size (the HBM
 * evaluation cache, which changes no result), device_games (concurrent searches; 0 = min(n, the model's max_batch);
 * more than max_batch is ERANGE), device_tree_kwords and device_waves_in_flight as in self-play.  Everything else is
 * ignored.
 * Errors: EINVAL for a bad FEN, an illegal move (the message names the position index), a FEN for hex or tic-tac-toe,
 * non-zero prior_noise_epsilon or a model of another game; ERANGE when a search runs out of tree memory (raise
 * device_tree_kwords or lower device_games).  The message is cattus_b200_last_error(). */
int cattus_b200_analyse(cattus_b200_t* model, const cattus_b200_selfplay_cfg* cfg, uint32_t n, const char* const* fens, const uint16_t* moves,
                        const uint32_t* move_offsets, cattus_b200_analysis_t** out);

/* Options of cattus_b200_analyse_opts.  struct_size must be sizeof(cattus_b200_analysis_opts). */
typedef struct cattus_b200_analysis_opts {
    uint32_t struct_size;
    uint32_t search_batch; /* descents per minibatch under virtual loss (DESIGN.md section 15); 0 or 1: one leaf in flight */
} cattus_b200_analysis_opts;

/* cattus_b200_analyse with options; opts NULL is cattus_b200_analyse.  With search_batch L > 1 every search runs
 * minibatches of L descents of its tree under virtual loss, so that the evaluator sees up to L leaves of one tree at
 * once: the mode for searching one position, or a few, deeply.  Its results are deterministic -- they depend on the
 * position, its history, the network, sim_num, explore_factor and L alone -- but are not those of one leaf in flight.
 * device_games 0 means min(n, max_batch / L); device_games x L above the model's max_batch is ERANGE, a bad
 * opts->struct_size EINVAL. */
int cattus_b200_analyse_opts(cattus_b200_t* model, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_analysis_opts* opts, uint32_t n,
                             const char* const* fens, const uint16_t* moves, const uint32_t* move_offsets, cattus_b200_analysis_t** out);

int cattus_b200_analysis_count(const cattus_b200_analysis_t* r, uint32_t* n);
int cattus_b200_analysis_get(const cattus_b200_analysis_t* r, uint32_t k, cattus_b200_analysis_position* out);
/* The root's children in edges() order (newest first, the order calc_moves_probabilities lists them): move, visits
 * (simulations_n), W (score_w, from the side to move at the root) and prior (init_score).  Any output may be NULL;
 * cap must hold n_children. */
int cattus_b200_analysis_children(const cattus_b200_analysis_t* r, uint32_t k, uint16_t* moves, uint32_t* visits, float* w, float* priors,
                                  uint32_t cap);
/* The principal variation: from the root, repeatedly the most visited child (equal counts: the one best_move's rule
 * picks), until a node that was never expanded or 16 plies. */
int cattus_b200_analysis_pv(const cattus_b200_analysis_t* r, uint32_t k, uint16_t* pv, uint32_t cap);
/* Minibatches the search of position k ran and its descents that were collisions (ended on a leaf an earlier descent
 * of the same minibatch had claimed).  One leaf in flight: minibatches = simulations, collisions 0.  Not searched: 0, 0.
 * Either output may be NULL. */
int cattus_b200_analysis_batches(const cattus_b200_analysis_t* r, uint32_t k, uint32_t* minibatches, uint32_t* collisions);
void cattus_b200_analysis_free(cattus_b200_analysis_t* r);

#ifdef __cplusplus
}
#endif
#endif /* CATTUS_B200_ANALYSIS_H */
