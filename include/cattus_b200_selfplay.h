/* cattus_b200_selfplay.h -- C ABI of the self-play driver that feeds the B200 evaluator (SURVEY.md section 8f-1/3).
 *
 * This is the CALLER side of the hot path: the reference's `MctsPlayer` (engine/src/mcts/mod.rs:105-454), the Hex and
 * TicTacToe rules it needs (engine/src/hex/core.rs:112-335, engine/src/ttt/core.rs:101-246), `NNetwork::evaluate`'s
 * flip + `ValueFuncCache` (engine/src/net/mod.rs:74-87,158-182; engine/src/mcts/cache.rs:31-75), the self-play game
 * loop (training/self-play/src/self_play.rs:94-276) and the `.traindata` writers (self_play.rs:33-61,
 * serialize/hex.rs:16-28, serialize/ttt.rs:17-22, serialize/chess.rs:18-57), restated in C++ so that "self-play MCTS
 * sims/s" can be measured without a Rust toolchain.  Chess (engine/src/chess/core.rs, threefold repetition through
 * MctsPlayer::detect_repetition, mcts/mod.rs:133-154) runs on the rules of cattus_b200/csrc/chess_rules.hpp, a
 * restatement of the third-party crate `chess` the reference uses (see include/cattus_b200_chess.h).
 *
 * What differs from the reference, on purpose: a worker thread there owns ONE tree with one leaf in flight, so the
 * evaluator never sees more than `threads` (<= 16) positions at once.  Here each worker thread advances
 * `games_per_thread` independent games as state machines; every game still runs its simulations strictly in the
 * reference's order (one leaf in flight per tree, so move choices are unchanged), but the leaves of all games of a
 * worker (or of one of its slot groups, `groups_per_thread`) go to the GPU as ONE batch.  With `games_per_thread = 1` and `leaf_queue = 1` it degenerates to the
 * reference's arrangement: one blocking `cattus_b200_eval` per leaf, batched across threads by the pinned queue.
 *
 * Randomness: the reference draws Dirichlet noise and temperature samples from the unseeded thread-local
 * `rand::rng()`.  Here every game owns a SplitMix64 stream seeded from (seed, game index), so a run is reproducible
 * and independent of scheduling, thread count and batch composition (the evaluator is batch invariant).
 */
#ifndef CATTUS_B200_SELFPLAY_H
#define CATTUS_B200_SELFPLAY_H

#include <stddef.h>
#include <stdint.h>

#include "cattus_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Evaluator callback: same contract as cattus_b200_eval_batch with the handle replaced by `ctx`.  Mirrors the
 * pluggable `Arc<dyn ValueFunction<Game>>` of MctsParams (engine/src/mcts/mod.rs:72-79).  Positions arrive with
 * Player1 to move (already flipped); probabilities must come back compact in ascending nn index over the legal moves. */
typedef int (*cattus_b200_eval_fn)(void* ctx, const uint64_t* planes, const uint8_t* legal_bitmaps, uint32_t n,
                                   float* probs_out, size_t probs_cap, uint32_t* prob_offsets, float* values_out);

/* Mirrors the JSON config of the self-play executable (training/self-play/src/self_play_cmd.rs:34-53) plus its
 * command line (:14-31). */
typedef struct cattus_b200_selfplay_cfg {
    uint32_t struct_size;
    uint32_t game;       /* CATTUS_B200_GAME_HEX, _TTT or _CHESS */
    uint32_t board_size; /* hex: 2..11; ttt: 3; chess: 8 */
    /* mcts.* */
    uint32_t sim_num;
    float explore_factor;
    const uint32_t* temperature_moves; /* temperature_policy as in the JSON: n_temperatures (move_threshold, */
    const float* temperature_values;   /* temperature) pairs; the LAST pair's temperature is the tail value  */
    uint32_t n_temperatures;           /* (self_play_cmd.rs:69-72).  0 pairs = constant 1.0                  */
    float prior_noise_alpha;
    float prior_noise_epsilon;
    uint32_t cache_size; /* ValueFuncCache max entries per evaluator; 0 = no cache */
    /* threads / batching */
    uint32_t threads;          /* worker threads (config.threads) */
    uint32_t games_per_thread; /* concurrent games per worker thread (>= 1); not in the reference */
    uint32_t leaf_queue;       /* 1: single-position requests go through cattus_b200_eval (cross-thread pinned queue) */
    /* games */
    uint32_t games_num;        /* total games of the job (even, self_play.rs:100) */
    uint32_t first_game;       /* this call plays game indices first_game, first_game + game_stride, ... < games_num */
    uint32_t game_stride;      /* (multi-GPU partition: rank r of n plays r, r + n, ...; 0 is read as 1)             */
    uint64_t seed;
    /* output */
    const char* out_dir1; /* NULL: do not write .traindata files */
    const char* out_dir2;
    uint32_t keep_records; /* 1: keep every game's moves and data entries in memory for the accessors below */
    uint32_t groups_per_thread; /* slot groups per worker, each with its own batch in flight while the worker simulates
                                 * the next group (0 or 1 = one group; > 1 needs the B200 evaluator) */
    uint32_t max_moves; /* 0 (the reference): play every game to its end.  > 0: stop a game after this many moves and
                         * record it as a draw -- for benches and tools that need a bounded amount of work */
    uint32_t speculate; /* needs cache_size > 0.  A device batch of 1 ... 256 positions costs the same time, so while leaves wait
                         * for the network, up to this many more positions per game ride in the same evaluator call and land
                         * in the cache: the best-scoring unvisited alternatives along the path just walked and the
                         * best-prior children of nodes expanded before.  Every search is unchanged (the cache returns what a
                         * fresh evaluation would); only batches below 192 rows are topped up.  For the UCI search and for
                         * trainer-sized jobs (a hundred games over a few threads); 0 = off, as the reference */
    uint32_t device_games; /* > 0: DEVICE-RESIDENT search (needs the B200 evaluator).  This many games run concurrently with
                            * their search trees in HBM, one warp per game: select, expansion and backpropagation run on
                            * the GPU, leaves go straight into the evaluator's device batch, and the host only acts once per
                            * MOVE (move choice, Dirichlet sample, game status, .traindata).  Same games, move for move and
                            * byte for byte, as the host-tree driver; threads / games_per_thread / cache_size / speculate /
                            * leaf_queue are ignored.  Must not exceed the evaluator's max_batch.  0 = trees on the host */
    uint32_t device_tree_kwords;     /* per tree buffer, in 1024 32-bit words; 0 = sized from sim_num and the free memory */
    uint32_t device_waves_in_flight; /* select -> evaluate -> expand rounds queued ahead of the host; 0 = 2 */
} cattus_b200_selfplay_cfg;

/* Mirrors the summary file (self_play_cmd.rs:131-149) and the metric keys the trainer reads
 * (training/cattus_train/train_process.py:176-186). */
typedef struct cattus_b200_selfplay_summary {
    uint32_t player1_wins, player2_wins, draws, games;
    uint64_t simulations;   /* develop_tree iterations (leaf selections) over all searches */
    uint64_t searches;      /* calc_moves_probabilities calls (= positions written) */
    uint64_t evaluations;   /* positions sent to the evaluator (cache misses) */
    uint64_t cache_hits;    /* cache.hits */
    uint64_t cache_misses;  /* cache.misses */
    uint64_t batches;       /* evaluator calls */
    uint64_t terminal_leaves;
    double seconds;         /* wall clock of the whole call */
    double search_duration; /* RunningAverage(0.99) of per-search seconds: mcts.search_duration */
    double eval_wait_seconds; /* summed over workers: time blocked in the evaluator */
    uint64_t speculative_evaluations; /* of `evaluations`: positions evaluated ahead into the cache (cfg.speculate) */
} cattus_b200_selfplay_summary;

typedef struct cattus_b200_selfplay cattus_b200_selfplay_t;

/* Plays the games with the B200 evaluator(s): player1 uses `model1`, player2 `model2` (may be the same handle or
 * NULL for "same", as when --model1-path == --model2-path, self_play_cmd.rs:93-106).  Blocks until all games of this
 * partition are finished.  The result object carries the summary and, if cfg->keep_records, the per-game records. */
int cattus_b200_selfplay_run(cattus_b200_t* model1, cattus_b200_t* model2, const cattus_b200_selfplay_cfg* cfg,
                             cattus_b200_selfplay_t** out);

/* The same driver over arbitrary evaluators (the reference's trait object).  Used by the CPU tests, which bind a
 * deterministic value function, and by the bench's CPU-baseline leg. */
int cattus_b200_selfplay_run_with(cattus_b200_eval_fn eval1, void* ctx1, cattus_b200_eval_fn eval2, void* ctx2,
                                  const cattus_b200_selfplay_cfg* cfg, cattus_b200_selfplay_t** out);

/* Options of cattus_b200_selfplay_run_opts (struct_size = sizeof, checked for equality: EINVAL otherwise). */
typedef struct cattus_b200_selfplay_opts {
    uint32_t struct_size;
    uint32_t search_batch; /* descents per minibatch under virtual loss (DESIGN.md sections 15 and 16); 0 or 1: one leaf in flight */
} cattus_b200_selfplay_opts;

/* cattus_b200_selfplay_run with options; opts NULL is cattus_b200_selfplay_run.  With search_batch L > 1 every search of
 * both models runs in minibatches: L descents in order on a frozen tree under virtual loss, then their leaves are
 * evaluated together and backed up in descent order, so that a few games fill the evaluator's batch.  Such games are
 * deterministic but are NOT the reference's games (a minibatched search is not MctsPlayer's); each game's random stream,
 * the temperature policy, root noise, tree reuse, repetition, max_moves and the .traindata format are unchanged, and
 * `simulations` still counts sim_num per search.  L > 1 needs the device-resident search (device_games > 0: EINVAL
 * otherwise); device_games x L above either model's max_batch is ERANGE. */
int cattus_b200_selfplay_run_opts(cattus_b200_t* model1, cattus_b200_t* model2, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_selfplay_opts* opts,
                                  cattus_b200_selfplay_t** out);

int cattus_b200_selfplay_summary_get(const cattus_b200_selfplay_t* r, cattus_b200_selfplay_summary* out);
/* Over all searches of the call: rounds of descents (one leaf in flight: one per simulation) and descents that ended on
 * a leaf an earlier descent of their minibatch had claimed (not simulations; 0 with one leaf in flight). */
int cattus_b200_selfplay_batches(const cattus_b200_selfplay_t* r, uint64_t* minibatches, uint64_t* collisions);
/* Number of games played by this call and, for the k-th of them (k in 0..n), its index / winner (0 none, 1, 2)
 * / move count. */
int cattus_b200_selfplay_game_count(const cattus_b200_selfplay_t* r, uint32_t* n);
int cattus_b200_selfplay_game_info(const cattus_b200_selfplay_t* r, uint32_t k, uint32_t* game_idx, uint32_t* winner,
                                   uint32_t* n_moves);
/* moves_out[n_moves]: the move indices (row * S + col) played (hex, tic-tac-toe). */
int cattus_b200_selfplay_game_moves(const cattus_b200_selfplay_t* r, uint32_t k, uint8_t* moves_out, uint32_t cap);
/* The same for any game; chess moves are from | to << 6 | promotion << 12 in real board coordinates
 * (include/cattus_b200_chess.h). */
int cattus_b200_selfplay_game_moves16(const cattus_b200_selfplay_t* r, uint32_t k, uint16_t* moves_out, uint32_t cap);
/* The exact bytes of `{game_idx:08}_{pos_idx:03}.traindata` and which out_dir (1 or 2) it belongs to. */
int cattus_b200_selfplay_entry(const cattus_b200_selfplay_t* r, uint32_t k, uint32_t pos_idx, uint8_t* bytes_out,
                               size_t cap, size_t* n_bytes, uint32_t* out_dir);
void cattus_b200_selfplay_free(cattus_b200_selfplay_t* r);

/* ---- one chess search at a time: the player behind the reference's UCI loop (engine/src/chess/uci.rs) ----
 * create = `ucinewgame` (MctsPlayer::new, uci.rs:59); the mcts.* fields, cache_size and seed of cfg are used.
 * go     = `position ...` + `go` (uci.rs:76-93, :158-161): the history is the FEN's position (NULL: the start position)
 *          followed by one position per move (the cache holds at most 128 Ki entries here); GamePlayer::next_move(pos_history) (mcts/mod.rs:448-454) searches with one
 *          leaf in flight (per-leaf cattus_b200_eval), reusing the tree of the previous `go` when the new position is
 *          in it (mod.rs:335-352).  Moves are from | to << 6 | promotion << 12 in real board coordinates
 *          (include/cattus_b200_chess.h). */
typedef struct cattus_b200_chess_search cattus_b200_chess_search_t;
typedef struct cattus_b200_chess_search_stats {
    uint32_t struct_size;
    uint32_t root_children;  /* legal moves of the searched position */
    uint32_t best_visits;    /* simulations that went through the most visited root child */
    uint32_t speculative_evaluations; /* of `evaluations`: positions evaluated ahead into the cache (cfg.speculate) */
    uint64_t simulations, evaluations, cache_hits, terminal_leaves; /* of this search */
    double seconds;
} cattus_b200_chess_search_stats;
int cattus_b200_chess_search_create(cattus_b200_t* model, const cattus_b200_selfplay_cfg* cfg, cattus_b200_chess_search_t** out);
int cattus_b200_chess_search_create_with(cattus_b200_eval_fn eval, void* ctx, const cattus_b200_selfplay_cfg* cfg,
                                         cattus_b200_chess_search_t** out);
int cattus_b200_chess_search_go(cattus_b200_chess_search_t* s, const char* fen, const uint16_t* moves, uint32_t n_moves,
                                uint16_t* best_move, cattus_b200_chess_search_stats* stats);
void cattus_b200_chess_search_destroy(cattus_b200_chess_search_t* s);
/* thread-local message of the last failed cattus_b200_selfplay_* call on this thread */
const char* cattus_b200_selfplay_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* CATTUS_B200_SELFPLAY_H */
