// Host runtime of the evaluator: weight blob -> device layouts, per-stream batch buffers ("lanes"), the launch
// sequence for one batch (captured into a CUDA graph per batch-size bucket), the pinned batch queue that the
// blocking per-leaf `eval` feeds, and metrics.  Everything here sits below the C ABI in include/cattus_b200.h.
//
// What it replaces in the reference (paths relative to /root/reference):
//   Model::new / Model::run          engine/src/net/model.rs:61-144, :146-218   -> Engine::Engine / run_bucket
//   Batcher::apply                   engine/src/util/batch.rs:49-177            -> Engine::eval_leaf + evaluator_loop
//   NNetwork::run_net metrics        engine/src/net/mod.rs:41-72                -> Engine::note_batch
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdint>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../../include/cattus_b200.h"
#include "kernels.cuh"
#include "tc_gemm.cuh"
#include "trunk_fused.cuh"
#include "trunk_small.cuh"

namespace cb2 {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define CB2_CUDA(expr)                                                                                        \
    do {                                                                                                      \
        cudaError_t e_ = (expr);                                                                              \
        if (e_ != cudaSuccess)                                                                                \
            throw ::cb2::Error(CATTUS_B200_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(e_) + " (" + \
                                                      __FILE__ + ":" + std::to_string(__LINE__) + ")");       \
    } while (0)

struct NetDims {
    uint32_t game = 0, s = 0, c_in = 0, moves = 0, f = 0, r = 0, vh = 0, ph = 0, hidden = 128;
    uint32_t arch = 0;  // 0: ConvNetV1 (net_utils.py:45-89); 1: SimpleTwoHeadedModel (net_utils.py:92-121; f, r, vh, ph unused)
    uint32_t features() const { return c_in * s * s; }  // SimpleTwoHeadedModel's width (net_utils.py:97-99)
    uint32_t s2() const { return s * s; }
    uint32_t wpp() const { return (s * s + 63) / 64; }
    uint32_t bitmap_bytes() const { return (moves + 7) / 8; }
};

// .cb2 weight blob (written by cattus_b200/export.py): 64-byte header + BN-folded fp32 tensors in PyTorch layouts.
struct Blob {
    NetDims d;
    std::vector<float> data;
    struct Conv {
        size_t w = 0, b = 0;  // offsets (in floats) into data
        uint32_t co = 0, ci = 0, k = 0;
    };
    Conv stem;
    std::vector<Conv> block_conv;  // 2 per block
    Conv vconv, pconv;
    size_t vfc1_w = 0, vfc1_b = 0, vfc2_w = 0, vfc2_b = 0, pfc_w = 0, pfc_b = 0;
    size_t d1_w = 0, d1_b = 0, d2_w = 0, d2_b = 0;  // SimpleTwoHeadedModel: _dense1, _dense2 (value head = vfc2_*, policy head = pfc_*)
    static Blob parse(const void* bytes, size_t n);
};

struct Op {
    int stage = 0;  // 0 encode, 1 trunk, 2 heads, 3 tail
    const char* name = "";
    std::function<void(cudaStream_t)> launch;
};

struct DeviceBuf {
    void* p = nullptr;
    size_t bytes = 0;
    void alloc(size_t n);  // zero-initialised
    void free_();
    template <class T>
    T* as() const { return static_cast<T*>(p); }
};

// One evaluator stream with everything a batch needs: pinned I/O blocks, device I/O blocks, activations, graphs.
struct Lane {
    int index = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    // pinned host
    uint8_t* h_in = nullptr;    // [16 B header: n][records]; swapped with the queue's open block
    float* h_values = nullptr;  // [max_batch]
    float* h_probs = nullptr;   // [max_batch * moves]
    float* zc_values = nullptr; // device-side aliases of h_values / h_probs (mapped pinned memory): small batches write
    float* zc_probs = nullptr;  // their outputs straight to the host, which takes two D2H copies off the critical path
    // device
    DeviceBuf d_in;  // same layout as h_in
    DeviceBuf d_values, d_probs;
    DeviceBuf d_x;       // bf16: encoded input NHWC [rows][64]; fp32: NCHW f32
    DeviceBuf d_act[3];  // trunk activations
    DeviceBuf d_hv, d_hp;  // head conv outputs
    DeviceBuf d_hidden;    // value FC1 output [max_batch][128] f32
    DeviceBuf d_logits;    // [max_batch][ld_logits] f32
    DeviceBuf d_dense;     // run_dense / encode staging (f32 NCHW)
    bool device_out = false;  // outputs stay in d_values / d_probs whatever the batch size (device-resident search)
    std::map<uint32_t, std::vector<Op>> ops;     // key: bucket | (dense_input << 31) | (device_out << 30)
    std::map<uint32_t, cudaGraphExec_t> graphs;  // same key
    // asynchronous batch in flight on this lane (eval_batch_submit .. eval_batch_wait)
    uint32_t async_n = 0, async_total = 0;
    std::vector<uint32_t> async_counts;
    std::chrono::steady_clock::time_point async_t0;
};

// A few helper threads that split the host-side packing of a large `eval_batch` chunk (memcpy + popcount per record)
// so that the first chunk reaches the GPU sooner and the host keeps ahead of a fast evaluator.
class PackPool {
  public:
    explicit PackPool(unsigned helpers);
    ~PackPool();
    // fn(slice) for slice in [0, slices); the caller takes part; returns false (nothing run) if the pool is busy
    bool try_run(int slices, const std::function<void(int)>& fn);

  private:
    void worker();
    std::vector<std::thread> threads_;
    std::mutex mu_, run_mu_;
    std::condition_variable cv_, done_cv_;
    const std::function<void(int)>* job_ = nullptr;
    int slices_ = 0, remaining_ = 0, active_ = 0;
    std::atomic<int> next_{0};
    uint64_t gen_ = 0;
    bool stop_ = false;
};

struct LeafRequest {
    float* probs_out;
    uint32_t probs_cap;
    uint32_t* n_probs;
    float* value_out;
    uint32_t count = 0;  // legal moves of this leaf
    int status = 1;      // 1 = pending, 0 = ok, <0 = error
    std::string error;
    std::atomic<int> done{0};  // set (release) after status / outputs are written: callers spin on it before sleeping
};

class Engine {
  public:
    Engine(const cattus_b200_desc& desc, const void* blob, size_t blob_bytes);
    ~Engine();

    void get_info(cattus_b200_info* info) const;
    void get_metrics(cattus_b200_metrics* m) const;

    void eval_leaf(const uint64_t* planes, const uint8_t* legal, LeafRequest* req);  // blocking
    void eval_batch(const uint64_t* planes, const uint8_t* legal, uint32_t n, float* probs_out, size_t probs_cap,
                    uint32_t* prob_offsets, float* values_out);
    // split form of eval_batch for one device batch (n <= max_batch): submit returns a ticket (the lane) or -1 when
    // `block` is false and every lane is busy; wait blocks, writes the outputs and frees the lane
    int eval_batch_submit(const uint64_t* planes, const uint8_t* legal, uint32_t n, bool block);
    void eval_batch_wait(int ticket, float* probs_out, size_t probs_cap, uint32_t* prob_offsets, float* values_out);
    void encode(const uint64_t* planes, uint32_t n, uint32_t batch, float* nchw_out);
    void run_dense(const float* nchw, uint32_t n, float* logits_out, float* values_out);
    void resident_upload(const uint64_t* planes, const uint8_t* legal, uint32_t n);
    void eval_resident(uint32_t n, cudaStream_t stream);
    void resident_download(uint32_t n, float* probs_out, size_t probs_cap, uint32_t* prob_offsets, float* values_out);
    void time_stage(uint32_t stage, uint32_t n, uint32_t iters, float* ms_out);
    void time_stages_split(uint32_t n, uint32_t iters, float* ms_out);
    void time_sustained(const uint64_t* planes, const uint8_t* legal, uint32_t n, uint32_t n_batches, uint32_t iters, float* total_ms);

    // Device-resident callers (the search of dsearch.cuh): reserve a lane, write records straight into its device input
    // block, enqueue the evaluator's kernels on a stream of their own (capturable), read d_values / d_probs on the device.
    struct ResidentIo {
        int lane = -1;
        uint8_t* d_block = nullptr;  // [u32 n][12 B pad][record 0 prefix 8 B | planes | legal bitmap] ...
        float* d_values = nullptr;
        float* d_probs = nullptr;    // capacity max_batch * moves floats
        uint32_t rec_bytes = 0, plane_words = 0, max_batch = 0, moves = 0, kernels = 0;
    };
    ResidentIo resident_acquire(bool block = true);  // block == false: lane == -1 when every stream is taken
    void resident_enqueue(int lane, cudaStream_t stream);  // the max_batch bucket's launch sequence; rows read from the block
    void resident_release(int lane);
    void note_resident(uint64_t batches, uint64_t positions, uint64_t launches, double last_seconds);
    int device() const { return device_; }

  private:
    // setup
    void upload_weights(const Blob& blob);
    void init_lane(Lane& lane);
    uint32_t bucket_for(uint32_t n) const;
    bool zero_copy_out(const Lane& lane, uint32_t bucket, bool dense_input) const { return !dense_input && !lane.device_out && bucket <= 512; }
    std::vector<Op>& ops_for(Lane& lane, uint32_t bucket, bool dense_input);
    void build_ops_bf16(Lane& lane, uint32_t bucket, std::vector<Op>& ops, bool dense_input);
    void build_ops_fp32(Lane& lane, uint32_t bucket, std::vector<Op>& ops, bool dense_input);
    void build_ops_simple(Lane& lane, uint32_t bucket, std::vector<Op>& ops, bool dense_input);
    void add_tail_ops(Lane& lane, uint32_t bucket, std::vector<Op>& ops, bool dense_input, bool value_tail, bool policy_tail);
    void run_bucket(Lane& lane, uint32_t bucket, cudaStream_t stream, bool use_graph, bool dense_input);
    void throw_device_error(const char* where, cudaError_t e);

    // batch plumbing
    uint32_t pack_record(uint8_t* dst, const uint64_t* planes, const uint8_t* legal, uint32_t prob_offset) const;  // returns #legal
    void submit(Lane& lane, uint32_t n, uint32_t total_probs);  // H2D + graph + D2H + event (async)
    void finish(Lane& lane, uint32_t n);                         // wait + device error check + metrics
    Lane& acquire_lane();
    Lane* try_acquire_lane();
    void release_lane(Lane& lane);
    void evaluator_loop();
    void note_batch(uint32_t n, double seconds);

    // tensor maps
    CUtensorMap make_map_2d(const void* base, uint64_t inner, uint64_t rows, uint64_t row_stride_bytes, uint32_t box_rows);
    CUtensorMap make_map_conv(const void* base, uint32_t channels, uint32_t boards, uint32_t nb);
    Op make_tc_op(int stage, const char* name, const TcGemmParams& p, uint32_t m_tiles, uint32_t n_tiles);
    int tc_stages_for(uint32_t ctas, int num_kb, uint32_t rows) const;

    NetDims d_;
    cattus_b200_desc desc_{};
    int device_ = 0;
    int sm_count_ = 0;
    uint32_t max_batch_ = 0;
    uint32_t precision_ = 0;
    RecLayout rec_{};
    bool derive_legal_ = false;
    bool fused_trunk_ = false;  // S == 8 && F in {64, 128, 256}: whole-trunk kernel (trunk_fused.cuh)
    bool fp8_ = false;          // precision FP8: the whole-trunk kernel's e4m3 instantiation (only where fused_trunk_ holds)
    bool small_trunk_ = false;  // F == 16: whole trunk + head convs in one kernel (trunk_small.cuh)
    bool simple_ = false;       // SimpleTwoHeadedModel: three dense layers, no convolutions

    // derived layout constants (bf16 path)
    uint32_t cin_pad_ = 64;  // encoded-input channels (multiple of 64)
    uint32_t ca_ = 64;       // trunk activation channels (multiple of 64)
    uint32_t nb_ = 1;        // boards per 128-row tile
    uint32_t vhp_ = 16, php_ = 16;

    // weights on device
    struct GemmW {
        DeviceBuf w, b;
        uint32_t n_umma = 16, n_tiles = 1, k_pad = 64;
    };
    std::vector<GemmW> convs_;  // stem, then 2 per block (bf16: [Np][9*Cin_pad] cut into contiguous pre-swizzled smem stages, tile_b() in engine.cu; fp32: torch layout f32)
    GemmW vconv_, pconv_, vfc1_, pfc_;
    GemmW dense1_, dense2_;  // SimpleTwoHeadedModel
    DeviceBuf vfc2_w_;
    float vfc2_b_ = 0.0f;
    DeviceBuf fused_w_, fused_b_;  // trunk_fused.cuh weight images + biases
    DeviceBuf fused_s_;            // FP8: per-output-channel dequantisation factors, [layers + 1][F] like fused_b_
    DeviceBuf small_w_, small_b_;  // trunk_small.cuh weight image + biases
    DeviceBuf trace_;              // optional clock64 trace of trunk_small (CATTUS_B200_TRACE_TRUNK=1)
    uint32_t small_stem_kc_ = 1;

    std::vector<std::unique_ptr<Lane>> lanes_;
    std::vector<char> lane_busy_;
    std::mutex lane_mu_;
    std::condition_variable lane_cv_;

    // leaf queue: workers write their record straight into the open pinned block
    std::mutex q_mu_;
    std::condition_variable q_cv_, q_space_cv_, done_cv_;
    uint8_t* open_block_ = nullptr;  // pinned, same layout as Lane::h_in
    std::vector<LeafRequest*> open_reqs_;
    uint32_t open_total_ = 0;
    std::atomic<uint32_t> open_count_{0};  // open_reqs_.size(), readable without the lock (evaluators spin on it briefly)
    std::vector<std::thread> evaluators_;
    bool stopping_ = false;

    // error word (mapped pinned) written by kernels before a trap
    uint32_t* h_err_ = nullptr;
    uint32_t* d_err_ = nullptr;

    std::unique_ptr<PackPool> pack_pool_;
    std::vector<uint32_t> resident_offsets_;  // host copy of the resident batch's probability offsets

    // L2 flush scratch for time_stage
    DeviceBuf flush_;

    // metrics
    mutable std::mutex m_mu_;
    cattus_b200_metrics metrics_{};
    uint32_t kernels_per_batch_ = 0;

    // driver entry point
    void* encode_tiled_ = nullptr;
};

}  // namespace cb2
