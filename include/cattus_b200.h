/* cattus_b200.h -- C ABI of the B200-native (sm_100a) network evaluator for Cattus.
 *
 * This is the drop-in boundary for the one hot path of poja/Cattus: batched neural-network evaluation of MCTS
 * leaf positions.  It replaces everything *below* the engine's evaluator trait
 *
 *     trait ValueFunction<Game> { fn evaluate(&self, &Position) -> (Vec<(Move, f32)>, f32); }
 *                                                        (reference: engine/src/mcts/value_func.rs:1-11)
 *
 * i.e. the body of `NNetwork` (engine/src/net/mod.rs:14-104) from `position_to_planes` output onwards:
 * the cross-thread `Batcher` (engine/src/util/batch.rs:49-177), `planes_to_tensor` (net/mod.rs:121-156),
 * `Model::new` / `Model::run` (engine/src/net/model.rs:61-144, :146-218), the non-finite clamp (net/mod.rs:57-61)
 * and `calc_moves_probs` (net/mod.rs:106-119).  Flip / cache / move-order mapping stay on the caller's side
 * (see INTEGRATION.md for the Rust `impl ValueFunction<Game> for CudaNetwork<Game>` shim that binds these symbols).
 *
 * Conventions
 *   - plain pointers and sizes only; every function returns 0 on success or a negative CATTUS_B200_E* code,
 *     never throws across the boundary; `cattus_b200_last_error()` gives the thread-local message.
 *   - There is NO CPU fallback: `create` fails unless the device is compute capability 10.x.
 *   - Planes are the bitboards `position_to_planes` yields (hex: engine/src/hex/net.rs:14-24, chess:
 *     engine/src/chess/net/mod.rs:19-60, ttt: engine/src/ttt/net.rs:14-24) packed as little-endian u64 words,
 *     `words_per_plane = ceil(S*S/64)`, low word first -- exactly what the .traindata serializers write
 *     (training/self-play/src/serialize/hex.rs:16-28, chess.rs:18-57).  Bit h*S+w of plane c is cell (h, w).
 *   - Legal moves are a 1-bit-per-nn-index bitmap of ceil(M/8) bytes, bit i of byte i/8 (the layout
 *     serialize/chess.rs:34-41 stores).  NULL means "derive it": legal = plane[2] & ~(plane[0] | plane[1]),
 *     which is `legal_moves()` for hex (engine/src/hex/core.rs:297-305) and tic-tac-toe.
 *   - Probabilities come back compact: one f32 per legal move in ascending nn index; they sum to 1 over the legal
 *     moves (net/mod.rs:106-119).  Values are the network's tanh output for the position as given; the caller
 *     negates it if it flipped the position (net/mod.rs:166-182).
 */
#ifndef CATTUS_B200_H
#define CATTUS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CATTUS_B200_ABI_VERSION 1

/* error codes */
#define CATTUS_B200_OK 0
#define CATTUS_B200_EINVAL (-1)   /* bad argument / descriptor / blob */
#define CATTUS_B200_ENODEV (-2)   /* no sm_100 device: there is no CPU fallback */
#define CATTUS_B200_ECUDA (-3)    /* CUDA runtime / driver error */
#define CATTUS_B200_ENOMEM (-4)
#define CATTUS_B200_ERANGE (-5)   /* n > max_batch, output capacity too small */
#define CATTUS_B200_EDEVICE (-6)  /* a kernel reported a pipeline fault (bounded mbarrier wait expired) */

/* games (decides words per plane and the derived-legal rule) */
#define CATTUS_B200_GAME_TTT 0
#define CATTUS_B200_GAME_HEX 1
#define CATTUS_B200_GAME_CHESS 2

/* precision: replaces the serde-tagged `InferenceConfig` variant (engine/src/net/model.rs:17-25) */
#define CATTUS_B200_PRECISION_BF16 0       /* tcgen05 bf16 x bf16 -> fp32 accumulate */
#define CATTUS_B200_PRECISION_FP32_CHECK 1 /* CUDA-core fp32 everywhere; the <=1e-4 check mode */
/* Opt-in, never a default: the conv trunk (stem, residual blocks, both 1x1 head convs) on tcgen05 kind::f8f6f4, e4m3 x e4m3 ->
 * fp32 accumulate, in the whole-trunk kernel only.  Weights are quantised per output channel at load (amax -> 448, scale applied
 * in the epilogue); activations are cast to e4m3 (round to nearest even, saturating) without a scale; the residual stream, the
 * head convs' outputs, the head FCs and the softmax stay bf16 / fp32.  About 10x the bf16 path's error against fp32 on the
 * project's random-init nets; playing strength on a trained net is not measured.
 * `create` accepts it only where CATTUS_B200_TRUNK_FUSED applies -- 8x8 boards, 64 / 128 / 256 filters, <= 32 planes,
 * VH + PH <= 64 (each padded to 16), `flags` bit 0 clear -- and fails with CATTUS_B200_EINVAL otherwise (16-filter nets,
 * SimpleTwoHeadedModel, the forced per-layer path).  Such a handle reports precision 2 and trunk_path FUSED;
 * cattus_b200_run_dense on it returns CATTUS_B200_EINVAL (there is no dense-input FP8 path). */
#define CATTUS_B200_PRECISION_FP8 2

typedef struct cattus_b200 cattus_b200_t;

/* Mirrors `NNetwork::new(model_path, inference_cfg, batch_size, cache)` (engine/src/net/mod.rs:24-39):
 * model_path -> weights_path (a .cb2 blob written by cattus_b200.export), inference_cfg -> device/precision,
 * batch_size -> max_batch.  Architecture fields may be 0 ("take it from the blob"); non-zero values are checked. */
typedef struct cattus_b200_desc {
    uint32_t struct_size; /* sizeof(cattus_b200_desc) */
    uint32_t game;
    uint32_t board_size;      /* S */
    uint32_t planes;          /* C_in */
    uint32_t moves;           /* M */
    uint32_t filters;         /* F  (residual_filter_num) */
    uint32_t blocks;          /* R  (residual_block_num) */
    uint32_t value_channels;  /* VH */
    uint32_t policy_channels; /* PH */
    int32_t device;           /* CUDA ordinal */
    uint32_t max_batch;       /* positions per device batch (reference: engine.model.batch_size) */
    uint32_t n_streams;       /* evaluator streams, each with its own batch buffers and CUDA graphs (>=1) */
    uint32_t precision;       /* CATTUS_B200_PRECISION_* */
    uint32_t flags;           /* bit 0: force the per-layer kernels and the standalone tail kernels (the comparison path of the
                               * parity tests); bit 1: FAULT INJECTION for tests -- the first head GEMM tile of every batch never
                               * publishes its accumulator, so the kernel's bounded wait expires and the call fails with
                               * CATTUS_B200_EDEVICE (a device fault poisons the process's CUDA context: destroy the handle, and
                               * evaluate again from a new process); other bits 0 */
    const char* weights_path; /* may be NULL when create_from_memory is used */
} cattus_b200_desc;

/* Mirrors the metric keys the trainer reads from the self-play summary (`model.activation_count`,
 * `model.run_duration`: engine/src/net/mod.rs:35-36,66-69; training/cattus_train/train_process.py:176-186). */
typedef struct cattus_b200_metrics {
    uint64_t activation_count;  /* device batches run */
    uint64_t positions;         /* positions evaluated */
    double run_duration_last;   /* seconds, last batch, host clock around copy+graph+copy (what run_net times) */
    double run_duration_ema;    /* RunningAverage(0.99) of the above (engine/src/util/metric.rs:1-20) */
    double mean_batch_fill;     /* positions / (activation_count * max_batch) */
    uint64_t kernel_launches;   /* kernels launched by this handle (graph nodes counted per replay) */
} cattus_b200_metrics;

typedef struct cattus_b200_info {
    uint32_t game, board_size, planes, moves, filters, blocks, value_channels, policy_channels;
    uint32_t words_per_plane;    /* u64 words per plane */
    uint32_t legal_bitmap_bytes; /* ceil(M/8) */
    uint32_t max_batch, n_streams, precision;
    uint32_t sm_count;
    uint32_t kernels_per_batch;  /* kernel nodes in one captured batch graph */
    uint32_t trunk_path;         /* CATTUS_B200_TRUNK_*: which kernel family runs the stem + residual blocks of this handle */
} cattus_b200_info;

/* cattus_b200_info.trunk_path.  The whole-trunk kernels cover fixed shapes; every other net takes the per-layer kernel,
 * which is correct for any ConvNetV1 within the blob's limits but re-reads its activations through L2 (about 2.5x slower). */
#define CATTUS_B200_TRUNK_PER_LAYER 0 /* one tcgen05 implicit-GEMM launch per conv layer (tc_gemm.cuh); any shape */
#define CATTUS_B200_TRUNK_FUSED 1     /* trunk_fused.cuh: 8x8 boards, 64 / 128 / 256 filters, <= 32 planes, VH + PH <= 64 */
#define CATTUS_B200_TRUNK_SMALL 2     /* trunk_small.cuh: 16 filters, boards 3..11, <= 32 planes, VH + PH <= 32 */
#define CATTUS_B200_TRUNK_FP32 3      /* precision FP32_CHECK: CUDA-core fp32 loops (parity only) */
#define CATTUS_B200_TRUNK_DENSE 4     /* SimpleTwoHeadedModel (net_utils.py:92-121): no convolutions, three dense layers */

/* Replaces Model::new (engine/src/net/model.rs:61-144). */
int cattus_b200_create(const cattus_b200_desc* desc, cattus_b200_t** out);
int cattus_b200_create_from_memory(const cattus_b200_desc* desc, const void* blob, size_t blob_bytes, cattus_b200_t** out);
void cattus_b200_destroy(cattus_b200_t* h);
int cattus_b200_get_info(const cattus_b200_t* h, cattus_b200_info* info);

/* The per-leaf call: replaces `NNetwork::evaluate_impl` below `to_planes` (engine/src/net/mod.rs:89-103), i.e.
 * Batcher::apply (util/batch.rs:49-177) + planes_to_tensor + run_net + calc_moves_probs.  Thread-safe and blocking:
 * any number of MCTS worker threads may call it concurrently; requests meet in a pinned host batch queue that the
 * evaluator streams drain (whatever is pending, up to max_batch, goes out as one batch -- no 20 ms deadline).
 *   planes       [planes * words_per_plane] u64
 *   legal_bitmap [ceil(M/8)] bytes or NULL (derive)
 *   probs_out    capacity probs_cap floats; receives *n_probs values (ascending nn index)
 */
int cattus_b200_eval(cattus_b200_t* h, const uint64_t* planes, const uint8_t* legal_bitmap, float* probs_out,
                     uint32_t probs_cap, uint32_t* n_probs, float* value_out);

/* Synchronous whole batch from HOST buffers (benches, tests, and a Rust Batcher that wants to keep its own
 * rendezvous): n positions, any n >= 1 (split internally into max_batch chunks pipelined over the streams).
 *   planes        [n][planes * words_per_plane] u64
 *   legal_bitmaps [n][ceil(M/8)] bytes or NULL
 *   probs_out     capacity probs_cap floats, compact; position b owns [prob_offsets[b], prob_offsets[b+1])
 *   prob_offsets  [n + 1]
 *   values_out    [n]
 */
int cattus_b200_eval_batch(cattus_b200_t* h, const uint64_t* planes, const uint8_t* legal_bitmaps, uint32_t n,
                           float* probs_out, size_t probs_cap, uint32_t* prob_offsets, float* values_out);

/* Split form of eval_batch for ONE device batch (1 <= n <= max_batch), so that a caller can keep several batches in
 * flight: submit packs the positions into a free evaluator stream's pinned block and enqueues copy-in, graph and
 * copy-out; *ticket identifies the stream, or is -1 when `block` is 0 and every stream is busy (with `block` != 0 the
 * call waits for a free stream).  wait blocks until that batch is done, writes the same outputs as eval_batch
 * (prob_offsets has n + 1 entries) and frees the stream.  Every submitted ticket must be waited exactly once.
 * Used by the self-play driver: one group of games is simulated while another group's leaves are on the GPU. */
int cattus_b200_eval_batch_submit(cattus_b200_t* h, const uint64_t* planes, const uint8_t* legal_bitmaps, uint32_t n,
                                  int block, int32_t* ticket);
int cattus_b200_eval_batch_wait(cattus_b200_t* h, int32_t ticket, float* probs_out, size_t probs_cap,
                                uint32_t* prob_offsets, float* values_out);

/* Mirrors planes_to_tensor (engine/src/net/mod.rs:121-156) through the device encode kernel: writes the dense
 * f32 NCHW tensor [batch_size][planes][S][S]; rows >= n are zero.  Used by the bit-exact parity tests. */
int cattus_b200_encode(cattus_b200_t* h, const uint64_t* planes, uint32_t n, uint32_t batch_size, float* nchw_out);

/* Mirrors Model::run (engine/src/net/model.rs:146-218): dense f32 NCHW in, raw policy logits [n][M] and tanh
 * values [n] out (the two outputs "policy", "value" of training/cattus_train/self_play.py:139-148).  Runs the
 * handle's precision path; with FP32_CHECK it is the <=1e-4 comparison point for test_net_output-style parity. */
int cattus_b200_run_dense(cattus_b200_t* h, const float* nchw, uint32_t n, float* logits_out, float* values_out);

/* Device-resident variant used to time the kernels without PCIe: upload once, evaluate many times, download.
 * `stream` is a cudaStream_t (as void*) or NULL for the handle's own stream; eval_resident only enqueues. */
int cattus_b200_resident_upload(cattus_b200_t* h, const uint64_t* planes, const uint8_t* legal_bitmaps, uint32_t n);
int cattus_b200_eval_resident(cattus_b200_t* h, uint32_t n, void* stream);
int cattus_b200_resident_download(cattus_b200_t* h, uint32_t n, float* probs_out, size_t probs_cap,
                                  uint32_t* prob_offsets, float* values_out);
/* Times `iters` replays of one trunk layer / one named stage on the handle's stream with CUDA events (ms each).
 * stage: 0 = encode, 1 = stem+residual trunk, 2 = heads (1x1 convs + FCs), 3 = mask/softmax/tanh tail, 4 = all (the
 * captured graph); an L2 flush (256 MiB memset) precedes every iteration, outside the timed bracket.
 * stage 5: every iteration is one pass of the whole sequence with an event after each stage; ms_out holds 3 * iters
 * values [encode + trunk, heads, tail] that add up to the pass (no flush between the stages, as inside the graph). */
int cattus_b200_time_stage(cattus_b200_t* h, uint32_t stage, uint32_t n, uint32_t iters, float* ms_out);
/* Sustained throughput: n_batches distinct resident batches of n positions (planes [n_batches * n][...], one batch per
 * evaluator stream: n_batches <= n_streams), `iters` graph replays rotating over them back to back on one stream, one
 * pair of CUDA events around the lot -> *total_ms.  No L2 flush: the rotation keeps the inputs cold. */
int cattus_b200_time_sustained(cattus_b200_t* h, const uint64_t* planes, const uint8_t* legal_bitmaps, uint32_t n, uint32_t n_batches,
                               uint32_t iters, float* total_ms);

int cattus_b200_get_metrics(const cattus_b200_t* h, cattus_b200_metrics* out);
const char* cattus_b200_last_error(void);
uint32_t cattus_b200_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* CATTUS_B200_H */
