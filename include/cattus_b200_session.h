/* cattus_b200_session.h -- C ABI of persistent device search sessions (DESIGN.md section 17).
 *
 * A session owns one search tree on the device and searches it in minibatches of L >= 2 descents under virtual loss
 * (cattus_b200_analyse_opts' search_batch, DESIGN.md section 15).  The tree lives across searches: when the next search's
 * position is the previous root, one of its children or one of its grandchildren, that subtree is kept
 * (MctsPlayer::calc_moves_probabilities' rule, engine/src/mcts/mod.rs:335-362); otherwise the search starts from a fresh
 * root.  There is no root noise.  A search runs on a host thread of the session: `go` returns at once, `stop` ends it at
 * the next minibatch boundary, `info` reads how it stands, `wait` returns its result.
 *
 * A search with node budget N and minibatch cap m runs minibatches while fewer than N new simulations are done and
 * fewer than m minibatches have run, each of min(L, N - done) descents: fixed N and m give deterministic results, and
 * N = sim_num from a fresh root is cattus_b200_analyse_opts(search_batch = L) bit for bit.  A stop or a deadline ends the
 * search as if m had been the number of minibatches it completed (at least one); the result reports that number.
 */
#ifndef CATTUS_B200_SESSION_H
#define CATTUS_B200_SESSION_H

#include <stddef.h>
#include <stdint.h>

#include "cattus_b200.h"
#include "cattus_b200_analysis.h"
#include "cattus_b200_selfplay.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cattus_b200_session cattus_b200_session_t;

/* cattus_b200_session_wait: the timeout passed and the search is still running (not an error) */
#define CATTUS_B200_SESSION_RUNNING 1

/* Why a search ended (cattus_b200_session_stats::stop_reason) */
#define CATTUS_B200_STOP_NODES 1       /* its node budget is done */
#define CATTUS_B200_STOP_MINIBATCHES 2 /* its minibatch cap is reached */
#define CATTUS_B200_STOP_REQUEST 3     /* cattus_b200_session_stop */
#define CATTUS_B200_STOP_DEADLINE 4    /* its deadline passed */
#define CATTUS_B200_STOP_CAPACITY 5    /* the tree buffer might not hold another minibatch's new leaves */
#define CATTUS_B200_STOP_FINISHED 6    /* the position's game is over: nothing was searched */

typedef struct cattus_b200_session_opts {
    uint32_t struct_size;  /* sizeof(cattus_b200_session_opts) */
    uint32_t search_batch; /* L, descents per minibatch: >= 2 and at most the model's max_batch */
    uint32_t tree_kwords;  /* words of each tree buffer / 1024; 0 = the largest the 2^26-word tree address space allows */
} cattus_b200_session_opts;

typedef struct cattus_b200_session_limits {
    uint32_t struct_size; /* sizeof(cattus_b200_session_limits) */
    uint32_t nodes;       /* new simulations on top of the kept tree; 0 = no limit */
    uint32_t minibatches; /* 0 = no limit */
    uint32_t pad;
    uint64_t deadline_us; /* microseconds from the call on the host's steady clock; 0 = none */
} cattus_b200_session_limits;

/* How the running (or last) search stands, as of its latest reported minibatch. */
typedef struct cattus_b200_session_snapshot {
    uint32_t struct_size; /* sizeof(cattus_b200_session_snapshot) */
    uint32_t valid;       /* 0: no minibatch of this search reported yet (the fields below are zero) */
    uint32_t searching;   /* 1 while the search runs */
    uint32_t simulations; /* new simulations of this search */
    uint32_t minibatches;
    uint32_t collisions;
    uint16_t best_move;   /* as cattus_b200_analysis_position::best_move */
    uint16_t pv_len;
    float q;
    double seconds;       /* since go */
    uint16_t pv[16];
} cattus_b200_session_snapshot;

typedef struct cattus_b200_session_stats {
    uint32_t struct_size;   /* sizeof(cattus_b200_session_stats) */
    uint32_t stop_reason;   /* CATTUS_B200_STOP_* */
    uint32_t reused_visits; /* the root's visits kept from the previous search (0: fresh root) */
    uint32_t pad;
    double seconds;         /* from go to the end of the search */
} cattus_b200_session_stats;

/* Creates a session on `model` for cfg's game (cfg: game / board_size, mcts.explore_factor; prior_noise_epsilon must be
 * 0; cache_size as in analysis; device_waves_in_flight).  The session holds one evaluator lane of the model for its
 * lifetime and leaves the others to the handle's other entry points: a model created with n_streams < 2, or with no
 * free lane, is EINVAL.  L < 2 or above max_batch, a bad struct_size, or a tree_kwords below a few minibatches' worth
 * or beyond the tree address space is EINVAL. */
int cattus_b200_session_create(cattus_b200_t* model, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_session_opts* opts,
                               cattus_b200_session_t** out);
/* The position of the next search: fen (NULL: the initial position; chess only) and moves as in cattus_b200_analyse.
 * EINVAL names a bad FEN or an illegal move; EINVAL while a search runs. */
int cattus_b200_session_set_position(cattus_b200_session_t* s, const char* fen, const uint16_t* moves, uint32_t n);
/* The next search starts from a fresh root whatever its position (a new game). */
int cattus_b200_session_new_game(cattus_b200_session_t* s);
/* Starts a search of the position set last and returns at once.  EINVAL while a search runs, before any position, or for
 * a bad struct_size. */
int cattus_b200_session_go(cattus_b200_session_t* s, const cattus_b200_session_limits* limits);
/* Ends the running search at its next minibatch boundary; nothing when none runs.  Any thread may call it. */
int cattus_b200_session_stop(cattus_b200_session_t* s);
/* Non-blocking: the latest snapshot of the running (or last) search, and a request for a fresh one after the next
 * minibatch. */
int cattus_b200_session_info(cattus_b200_session_t* s, cattus_b200_session_snapshot* out);
/* Waits up to timeout_ms (UINT32_MAX: without limit) for the search to end.  Returns CATTUS_B200_SESSION_RUNNING when
 * it has not, else its result as a one-entry analysis (free it with cattus_b200_analysis_free; simulations counts the
 * search's new ones) or the error the search met (ERANGE for a tree path deeper than the path buffer).  After an
 * error the session stays usable: its next search starts from a fresh root. */
int cattus_b200_session_wait(cattus_b200_session_t* s, uint32_t timeout_ms, cattus_b200_analysis_t** result);
/* The session figures of a result of cattus_b200_session_wait. */
int cattus_b200_session_result_stats(const cattus_b200_analysis_t* r, cattus_b200_session_stats* out);
/* Stops a running search, joins the session's thread and frees everything. */
void cattus_b200_session_destroy(cattus_b200_session_t* s);

#ifdef __cplusplus
}
#endif
#endif /* CATTUS_B200_SESSION_H */
