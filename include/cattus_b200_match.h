/* cattus_b200_match.h -- C ABI of colour-balanced match play between two networks from an opening suite.
 *
 * The games run on the device-resident search of cattus_b200_selfplay_run's `device_games` mode (search trees in HBM,
 * one warp per tree), thousands at a time, with the self-play game loop unchanged: opening k is played twice, game
 * 2k with model A as player 1 and game 2k + 1 with model B as player 1 (the parity rule self-play uses for model1 /
 * model2).  Each game draws from its own SplitMix64 stream seeded from (cfg->seed, game index), takes the config's
 * temperature policy and root noise, reuses each player's tree between its own moves, ends in a draw on a threefold
 * repetition and is adjudicated a draw after cfg->max_moves moves (counted from the opening; 0 = no limit).
 *
 * Repetition checks, inside the search and in the game, look back into the opening's positions since the last pawn
 * move or capture (chess; hex and tic-tac-toe have no repetition).  The temperature policy counts moves from the
 * opening position, as if the game had started there.  So a match whose openings are all the initial position plays,
 * game for game, what cattus_b200_selfplay_run(A, B) plays with games_num = 2n and the same seed.  A game depends on its
 * opening, its colour, the networks, cfg and side_b alone -- not on device_games, device_waves_in_flight, the cache or
 * the other openings.  (With root noise or a non-zero temperature the opening's place k in the input matters too: the
 * random stream is seeded from the game index 2k + c.)
 */
#ifndef CATTUS_B200_MATCH_H
#define CATTUS_B200_MATCH_H

#include <stddef.h>
#include <stdint.h>

#include "cattus_b200.h"
#include "cattus_b200_selfplay.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cattus_b200_match cattus_b200_match_t;

/* What side B plays with where it differs from cfg (everything else is shared). */
typedef struct cattus_b200_match_side {
    uint32_t struct_size;
    uint32_t sim_num;     /* 0: cfg->sim_num; otherwise > 1 */
    float explore_factor; /* < 0: cfg->explore_factor */
} cattus_b200_match_side;

/* Points are counted for A: a win 1, a draw 1/2, a loss 0.  pairs[j]: the openings (game pairs) in which A scored j / 2
 * points over its two games -- the pentanomial counts. */
typedef struct cattus_b200_match_summary {
    uint32_t struct_size;
    uint32_t a_wins, b_wins, draws, games;
    uint32_t openings; /* n */
    uint32_t skipped;  /* openings whose position was already finished: not played, in no count */
    uint32_t pairs[5];
    uint64_t simulations; /* develop_tree iterations over all searches of both sides */
    uint64_t evaluations; /* positions sent to the evaluators */
    double seconds;       /* wall clock of the whole call */
} cattus_b200_match_summary;

enum {
    CATTUS_B200_MATCH_END_RULES = 1,      /* mate, stalemate, the fifty-move rule, insufficient material; hex / ttt: the rules */
    CATTUS_B200_MATCH_END_REPETITION = 2, /* threefold repetition: a draw */
    CATTUS_B200_MATCH_END_MAX_MOVES = 3,  /* cfg->max_moves reached: adjudicated a draw */
};

typedef struct cattus_b200_match_game {
    uint32_t struct_size;
    uint32_t opening;      /* index into the openings */
    uint32_t a_is_player1; /* 1 in game 2k, 0 in game 2k + 1 */
    uint32_t winner;       /* 0 draw, 1 / 2 that player (chess: white / black) */
    uint32_t termination;  /* CATTUS_B200_MATCH_END_* */
    uint32_t n_moves;      /* moves played from the opening position */
} cattus_b200_match_game;

/* Plays the 2n games of n openings between model_a and model_b (any precision each, FP8 included).  model_b NULL or
 * model_a means one handle: one evaluator and one cache, as in self-play.  The openings are given as in
 * cattus_b200_analyse: opening k is fens[k] (NULL or fens NULL: the initial position; chess only) followed by
 * moves[move_offsets[k] .. move_offsets[k + 1]) (move_offsets NULL: no moves).  An opening whose position is already
 * finished (a threefold repetition in its moves included) is reported with its status and not played.
 * cfg: game / board_size, mcts.* (sim_num, explore_factor, temperature_policy, prior noise), cache_size (the HBM
 * evaluation cache, which changes no game), seed, max_moves, device_games (concurrent games; 0 = min(2n, max_batch);
 * more than either model's max_batch is ERANGE), device_tree_kwords (sized from the larger sim_num when 0) and
 * device_waves_in_flight as in self-play.  games_num, first_game, game_stride, out_dir*, keep_records and the host-driver
 * fields are ignored.  side_b: NULL = the same settings for both sides.
 * Errors: EINVAL for a bad FEN or an illegal move (the message names the opening index), a FEN for hex or tic-tac-toe,
 * models of another game or on different devices, and sim_num < 2 on either side; ERANGE when a search runs out of tree
 * memory (raise device_tree_kwords or lower device_games).  The message is cattus_b200_last_error(). */
int cattus_b200_match_run(cattus_b200_t* model_a, cattus_b200_t* model_b, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_match_side* side_b,
                          uint32_t n, const char* const* fens, const uint16_t* moves, const uint32_t* move_offsets, cattus_b200_match_t** out);

/* Options of cattus_b200_match_run_opts (struct_size = sizeof, checked for equality: EINVAL otherwise). */
typedef struct cattus_b200_match_opts {
    uint32_t struct_size;
    uint32_t search_batch_a; /* descents per minibatch under virtual loss of A's searches (DESIGN.md section 16); 0 or 1: one leaf in flight */
    uint32_t search_batch_b; /* the same for B */
} cattus_b200_match_opts;

/* cattus_b200_match_run with options; opts NULL is cattus_b200_match_run.  A side with search_batch L > 1 searches in
 * minibatches of L descents under virtual loss (see cattus_b200_selfplay_run_opts): its games are deterministic but are
 * NOT the reference's games, so a match between L = 1 and L > 1 of the same net measures what the minibatches cost in
 * games.  device_games x the larger L above either model's max_batch is ERANGE; device_games 0 takes
 * min(2n, max_batch / the larger L). */
int cattus_b200_match_run_opts(cattus_b200_t* model_a, cattus_b200_t* model_b, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_match_side* side_b,
                               const cattus_b200_match_opts* opts, uint32_t n, const char* const* fens, const uint16_t* moves,
                               const uint32_t* move_offsets, cattus_b200_match_t** out);

int cattus_b200_match_summary_get(const cattus_b200_match_t* r, cattus_b200_match_summary* out);
/* side 0 = A, 1 = B (ERANGE otherwise): that side's rounds of descents over all its searches (one leaf in flight: one
 * per simulation) and its descents that collided with an earlier one of their minibatch. */
int cattus_b200_match_batches(const cattus_b200_match_t* r, uint32_t side, uint64_t* minibatches, uint64_t* collisions);
/* status of opening k: 0 played; 1 / 2 already won by that player, 3 already drawn -- not played */
int cattus_b200_match_opening_status(const cattus_b200_match_t* r, uint32_t k, uint32_t* status);
/* The games played, by game index (opening, then colour); summary.games of them. */
int cattus_b200_match_game_get(const cattus_b200_match_t* r, uint32_t k, cattus_b200_match_game* out);
/* moves[n_moves] of game k, in the game's encoding (chess from | to << 6 | promotion << 12 in real board coordinates,
 * include/cattus_b200_chess.h; hex and tic-tac-toe cell index). */
int cattus_b200_match_game_moves(const cattus_b200_match_t* r, uint32_t k, uint16_t* moves, uint32_t cap);
void cattus_b200_match_free(cattus_b200_match_t* r);

#ifdef __cplusplus
}
#endif
#endif /* CATTUS_B200_MATCH_H */
