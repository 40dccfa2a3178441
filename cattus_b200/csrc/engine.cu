// Engine implementation + the extern "C" boundary (include/cattus_b200.h).  Single translation unit: the kernels
// live in headers and are instantiated here.
#include "engine.hpp"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>

namespace cb2 {

static inline uint32_t round_up(uint32_t x, uint32_t m) { return (x + m - 1) / m * m; }
static inline uint32_t ceil_div(uint32_t x, uint32_t m) { return (x + m - 1) / m; }
static constexpr int kRecPrefix = 8;             // per-record [prob offset, #legal]
static constexpr int kRecs0 = 16 + kRecPrefix;  // byte offset of record 0's planes inside a batch block

// ------------------------------------------------------------------------------------------------ blob
static constexpr uint32_t kBlobMagic = 0x00324243u;  // "CB2\0"

Blob Blob::parse(const void* bytes, size_t n) {
    if (bytes == nullptr || n < 64) throw Error(CATTUS_B200_EINVAL, "weight blob too small");
    const uint32_t* h = static_cast<const uint32_t*>(bytes);
    if (h[0] != kBlobMagic) throw Error(CATTUS_B200_EINVAL, "weight blob: bad magic (expected CB2)");
    if (h[1] != 1) throw Error(CATTUS_B200_EINVAL, "weight blob: unsupported version");
    Blob b;
    b.d.game = h[2];
    b.d.s = h[3];
    b.d.c_in = h[4];
    b.d.moves = h[5];
    b.d.f = h[6];
    b.d.r = h[7];
    b.d.vh = h[8];
    b.d.ph = h[9];
    b.d.hidden = h[10];
    b.d.arch = h[11];
    if (b.d.arch == 1) {
        // SimpleTwoHeadedModel (net_utils.py:92-121): dense1 w[n,n] b[n] | dense2 w b | value w[n] b[1] | policy w[M,n] b[M]
        NetDims& s = b.d;
        const size_t nf = s.features();
        if (s.game > 2 || s.s < 2 || s.s > 11 || s.c_in == 0 || s.c_in > 64 || s.moves == 0 || s.moves > 4096 || s.f || s.r || s.vh || s.ph || s.hidden != nf)
            throw Error(CATTUS_B200_EINVAL, "weight blob: SimpleTwoHeadedModel header out of the supported range");
        size_t off = 0;
        auto take = [&](size_t cnt) {
            size_t o = off;
            off += cnt;
            return o;
        };
        b.d1_w = take(nf * nf);
        b.d1_b = take(nf);
        b.d2_w = take(nf * nf);
        b.d2_b = take(nf);
        b.vfc2_w = take(nf);
        b.vfc2_b = take(1);
        b.pfc_w = take(static_cast<size_t>(s.moves) * nf);
        b.pfc_b = take(s.moves);
        if (n != 64 + off * sizeof(float))
            throw Error(CATTUS_B200_EINVAL, "weight blob: size " + std::to_string(n) + " does not match its SimpleTwoHeadedModel header (expected " +
                                                std::to_string(64 + off * sizeof(float)) + ")");
        b.data.resize(off);
        std::memcpy(b.data.data(), static_cast<const uint8_t*>(bytes) + 64, off * sizeof(float));
        for (float v : b.data)
            if (!std::isfinite(v)) throw Error(CATTUS_B200_EINVAL, "weight blob: non-finite weight");
        return b;
    }
    if (b.d.arch != 0) throw Error(CATTUS_B200_EINVAL, "weight blob: unknown architecture tag");
    const NetDims& d = b.d;
    if (d.game > 2 || d.s < 2 || d.s > 11 || d.c_in == 0 || d.c_in > 64 || d.moves == 0 || d.moves > 4096 || d.f == 0 ||
        d.f > 256 || d.vh == 0 || d.vh > 64 || d.ph == 0 || d.ph > 64 || d.hidden != 128 || d.r > 64)
        throw Error(CATTUS_B200_EINVAL, "weight blob: architecture out of the supported range");
    size_t off = 0;
    auto take = [&](size_t cnt) {
        size_t o = off;
        off += cnt;
        return o;
    };
    auto conv = [&](uint32_t co, uint32_t ci, uint32_t k) {
        Conv c;
        c.co = co;
        c.ci = ci;
        c.k = k;
        c.w = take(static_cast<size_t>(co) * ci * k * k);
        c.b = take(co);
        return c;
    };
    const uint32_t s2 = d.s2();
    b.stem = conv(d.f, d.c_in, 3);
    for (uint32_t i = 0; i < 2 * d.r; ++i) b.block_conv.push_back(conv(d.f, d.f, 3));
    b.vconv = conv(d.vh, d.f, 1);
    b.vfc1_w = take(static_cast<size_t>(d.hidden) * d.vh * s2);
    b.vfc1_b = take(d.hidden);
    b.vfc2_w = take(d.hidden);
    b.vfc2_b = take(1);
    b.pconv = conv(d.ph, d.f, 1);
    b.pfc_w = take(static_cast<size_t>(d.moves) * d.ph * s2);
    b.pfc_b = take(d.moves);
    if (n != 64 + off * sizeof(float))
        throw Error(CATTUS_B200_EINVAL, "weight blob: size " + std::to_string(n) + " does not match its header (expected " +
                                            std::to_string(64 + off * sizeof(float)) + ")");
    b.data.resize(off);
    std::memcpy(b.data.data(), static_cast<const uint8_t*>(bytes) + 64, off * sizeof(float));
    for (float v : b.data)
        if (!std::isfinite(v)) throw Error(CATTUS_B200_EINVAL, "weight blob: non-finite weight");
    return b;
}

// ------------------------------------------------------------------------------------------------ buffers
void DeviceBuf::alloc(size_t n) {
    free_();
    bytes = std::max<size_t>(n, 256);
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
        p = nullptr;
        throw Error(CATTUS_B200_ENOMEM, std::string("cudaMalloc(") + std::to_string(bytes) + "): " + cudaGetErrorString(e));
    }
    CB2_CUDA(cudaMemset(p, 0, bytes));
}
void DeviceBuf::free_() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
}

static std::vector<__nv_bfloat16> to_bf16(const std::vector<float>& v) {
    std::vector<__nv_bfloat16> o(v.size());
    for (size_t i = 0; i < v.size(); ++i) o[i] = __float2bfloat16_rn(v[i]);
    return o;
}

// B operand image of tc_gemm: the [N_pad][K_pad] K-major matrix cut into the kernel's smem stages, each stage (n_umma rows x
// 64 k = 128 B per row) stored CONTIGUOUSLY and already in the 128-byte-swizzled order the UMMA descriptor reads (16-byte
// chunk c of row r sits at chunk c ^ (r & 7)), stages ordered [n_tile][k-block].  One stage is then ONE linear bulk copy
// (cp.async.bulk) instead of a tensor-map box of n_umma separate 128-byte rows: the producer thread of the policy FC spent
// ~300 cycles per box on those, 786 cycles per k-block at B = 1 whatever the ring depth (clock64 trace, DESIGN.md section 5).
template <class G>
static std::vector<float> tile_b(const std::vector<float>& w, const G& g) {
    const size_t num_kb = g.k_pad / 64, np = static_cast<size_t>(g.n_umma) * g.n_tiles;
    std::vector<float> t(w.size());
    for (size_t o = 0; o < np; ++o) {
        const size_t r = o % g.n_umma;
        for (size_t k = 0; k < g.k_pad; ++k) {
            const size_t c = (k % 64) / 8, e = k % 8;
            t[(((o / g.n_umma) * num_kb + k / 64) * g.n_umma + r) * 64 + ((c ^ (r & 7)) * 8 + e)] = w[o * g.k_pad + k];
        }
    }
    return t;
}
template <class T>
static void upload(DeviceBuf& buf, const std::vector<T>& v) {
    buf.alloc(v.size() * sizeof(T));
    CB2_CUDA(cudaMemcpy(buf.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
}

// ------------------------------------------------------------------------------------------------ construction
Engine::Engine(const cattus_b200_desc& desc, const void* blob_bytes, size_t blob_n) : desc_(desc) {
    Blob blob = Blob::parse(blob_bytes, blob_n);
    d_ = blob.d;
    auto chk = [&](uint32_t want, uint32_t have, const char* what) {
        if (want != 0 && want != have)
            throw Error(CATTUS_B200_EINVAL, std::string("descriptor ") + what + "=" + std::to_string(want) +
                                                " does not match the weight blob (" + std::to_string(have) + ")");
    };
    chk(desc.board_size, d_.s, "board_size");
    chk(desc.planes, d_.c_in, "planes");
    chk(desc.moves, d_.moves, "moves");
    simple_ = d_.arch == 1;
    chk(desc.filters, d_.f, "filters");
    chk(desc.blocks, d_.r, "blocks");
    chk(desc.value_channels, d_.vh, "value_channels");
    chk(desc.policy_channels, d_.ph, "policy_channels");
    if (desc.game != d_.game) throw Error(CATTUS_B200_EINVAL, "descriptor game does not match the weight blob");
    if (desc.max_batch == 0 || desc.max_batch > (1u << 16)) throw Error(CATTUS_B200_EINVAL, "max_batch must be in 1..65536");
    if (desc.precision > CATTUS_B200_PRECISION_FP8) throw Error(CATTUS_B200_EINVAL, "unknown precision");
    max_batch_ = desc.max_batch;
    precision_ = desc.precision;
    const uint32_t n_streams = std::max<uint32_t>(1, std::min<uint32_t>(desc.n_streams, 32));

    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        throw Error(CATTUS_B200_ENODEV, std::string("no CUDA device (") + cudaGetErrorString(e) + "); there is no CPU fallback");
    if (desc.device < 0 || desc.device >= count) throw Error(CATTUS_B200_ENODEV, "device ordinal out of range");
    device_ = desc.device;
    cudaDeviceProp prop{};
    CB2_CUDA(cudaGetDeviceProperties(&prop, device_));
    if (prop.major != 10)
        throw Error(CATTUS_B200_ENODEV, std::string("device ") + prop.name + " is compute capability " + std::to_string(prop.major) +
                                            "." + std::to_string(prop.minor) + "; this library contains sm_100a code only and has no fallback");
    CB2_CUDA(cudaSetDevice(device_));
    sm_count_ = prop.multiProcessorCount;

    // record layout shared by host packing and the kernels
    derive_legal_ = (d_.game != CATTUS_B200_GAME_CHESS);
    if (derive_legal_ && (d_.c_in < 3 || d_.moves != d_.s2()))
        throw Error(CATTUS_B200_EINVAL, "derived legality needs >= 3 planes and moves == S*S");
    rec_.planes = static_cast<int>(d_.c_in);
    rec_.wpp = static_cast<int>(d_.wpp());
    rec_.s = static_cast<int>(d_.s);
    rec_.moves = static_cast<int>(d_.moves);
    rec_.legal_words = static_cast<int>(ceil_div(d_.moves, 32));
    const int plane_bytes = rec_.planes * rec_.wpp * 8;
    rec_.legal_off = derive_legal_ ? -1 : plane_bytes;
    // each record is preceded by an 8-byte prefix [u32 offset of its probabilities in the compact output][u32 #legal]
    // written by the host while packing (it counts the legal moves anyway), so no device-side count + scan is needed
    rec_.rec_bytes = kRecPrefix + plane_bytes + (derive_legal_ ? 0 : static_cast<int>(round_up(static_cast<uint32_t>(rec_.legal_words) * 4, 8)));

    // bf16 layout constants
    cin_pad_ = round_up(d_.c_in, 64);
    ca_ = round_up(d_.f, 64);
    nb_ = std::max<uint32_t>(1, 128 / d_.s2());
    vhp_ = round_up(d_.vh, 16);
    php_ = round_up(d_.ph, 16);

    {
        cudaDriverEntryPointQueryResult q;
        CB2_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &encode_tiled_, cudaEnableDefault, &q));
        if (q != cudaDriverEntryPointSuccess || encode_tiled_ == nullptr)
            throw Error(CATTUS_B200_ECUDA, "cuTensorMapEncodeTiled is not available from this driver");
    }
    CB2_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&h_err_), 64, cudaHostAllocMapped));
    std::memset(h_err_, 0, 64);
    CB2_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&d_err_), h_err_, 0));
    CB2_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem_bytes(kTcStages)));
    CB2_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem_bytes(kTcStagesDeep)));
    CB2_CUDA(cudaFuncSetAttribute(tc_gemm_dual_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem_bytes(kTcStages)));
    CB2_CUDA(cudaFuncSetAttribute(tc_gemm_dual_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem_bytes(kTcStagesDeep)));
    // whole-trunk kernel: 8x8 boards, 128 filters (flags bit 0 forces the per-layer path, used by the parity tests)
    // FP8 exists only as an instantiation of this kernel: every other shape is refused rather than run in another precision
    fp8_ = precision_ == CATTUS_B200_PRECISION_FP8;
    const bool fused_shape = !simple_ && d_.s == 8 && (d_.f == 64 || d_.f == 128 || d_.f == 256) && d_.c_in <= 32 && d_.wpp() == 1 &&
                             (desc.flags & 1u) == 0 && (sm_count_ >= 2) && vhp_ + php_ <= 64;
    if (fp8_ && !fused_shape)
        throw Error(CATTUS_B200_EINVAL, "precision FP8 is only available on the whole-trunk kernel: ConvNetV1 with 8x8 boards, 64 / 128 / 256 filters, "
                                        "<= 32 input planes, value + policy head channels (each padded to 16) <= 64, and flags bit 0 clear; this net has S=" +
                                            std::to_string(d_.s) + " F=" + std::to_string(d_.f) + " C_in=" + std::to_string(d_.c_in) + " VH=" +
                                            std::to_string(d_.vh) + " PH=" + std::to_string(d_.ph) + (simple_ ? " (SimpleTwoHeadedModel)" : "") +
                                            ((desc.flags & 1u) ? " flags bit 0 set" : ""));
    fused_trunk_ = fused_shape && (precision_ == CATTUS_B200_PRECISION_BF16 || fp8_);
    if (fused_trunk_) {
        auto smem = [](auto kernel, int bytes) { CB2_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes)); };
        using B = __nv_bfloat16;
        using E8 = __nv_fp8_e4m3;
        if (d_.f == 64) fp8_ ? smem(trunk_fused_kernel<64, E8>, FtG<64, E8>::kSmemBytes) : smem(trunk_fused_kernel<64, B>, FtG<64, B>::kSmemBytes);
        if (d_.f == 128) fp8_ ? smem(trunk_fused_kernel<128, E8>, FtG<128, E8>::kSmemBytes) : smem(trunk_fused_kernel<128, B>, FtG<128, B>::kSmemBytes);
        if (d_.f == 256) fp8_ ? smem(trunk_fused_kernel<256, E8>, FtG<256, E8>::kSmemBytes) : smem(trunk_fused_kernel<256, B>, FtG<256, B>::kSmemBytes);
    }
    // 16-filter nets (every shipped training config): whole trunk + both head convs in one kernel
    small_trunk_ = !simple_ && precision_ == CATTUS_B200_PRECISION_BF16 && d_.f == 16 && d_.c_in <= 32 && d_.s >= 3 && d_.s <= 11 && vhp_ + php_ <= 32 &&
                   (desc.flags & 1u) == 0;
    if (small_trunk_) {
        small_stem_kc_ = ceil_div(d_.c_in, 16);
        CB2_CUDA(cudaFuncSetAttribute(trunk_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    }

    upload_weights(blob);

    for (uint32_t i = 0; i < n_streams; ++i) {
        lanes_.emplace_back(new Lane());
        lanes_.back()->index = static_cast<int>(i);
        init_lane(*lanes_.back());
    }
    lane_busy_.assign(n_streams, 0);
    const size_t in_bytes = kRecs0 + static_cast<size_t>(max_batch_) * rec_.rec_bytes;
    CB2_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&open_block_), in_bytes, cudaHostAllocDefault));
    std::memset(open_block_, 0, in_bytes);
    open_reqs_.reserve(max_batch_);

    // warm the most common graph so the first leaf does not pay for capture
    {
        Lane& l = *lanes_[0];
        *reinterpret_cast<uint32_t*>(l.h_in) = 0;
        CB2_CUDA(cudaMemcpyAsync(l.d_in.p, l.h_in, 16, cudaMemcpyHostToDevice, l.stream));
        run_bucket(l, bucket_for(max_batch_), l.stream, true, false);
        cudaError_t se = cudaStreamSynchronize(l.stream);
        if (se != cudaSuccess) throw_device_error("warm-up batch", se);
        kernels_per_batch_ = static_cast<uint32_t>(ops_for(l, bucket_for(max_batch_), false).size());
    }
    for (uint32_t i = 0; i < n_streams; ++i) evaluators_.emplace_back([this] { evaluator_loop(); });
    pack_pool_.reset(new PackPool(std::min(7u, std::max(1u, std::thread::hardware_concurrency() / 2))));
}

Engine::~Engine() {
    {
        std::lock_guard<std::mutex> g(q_mu_);
        stopping_ = true;
    }
    q_cv_.notify_all();
    q_space_cv_.notify_all();
    for (auto& t : evaluators_) t.join();
    pack_pool_.reset();
    cudaSetDevice(device_);
    cudaDeviceSynchronize();
    for (auto& lp : lanes_) {
        Lane& l = *lp;
        for (auto& kv : l.graphs) cudaGraphExecDestroy(kv.second);
        if (l.stream) cudaStreamDestroy(l.stream);
        if (l.done) cudaEventDestroy(l.done);
        if (l.h_in) cudaFreeHost(l.h_in);
        if (l.h_values) cudaFreeHost(l.h_values);
        if (l.h_probs) cudaFreeHost(l.h_probs);
        for (DeviceBuf* b : {&l.d_in, &l.d_values, &l.d_probs, &l.d_x, &l.d_act[0], &l.d_act[1], &l.d_act[2], &l.d_hv,
                             &l.d_hp, &l.d_hidden, &l.d_logits, &l.d_dense})
            b->free_();
    }
    if (open_block_) cudaFreeHost(open_block_);
    if (h_err_) cudaFreeHost(h_err_);
    for (auto& c : convs_) {
        c.w.free_();
        c.b.free_();
    }
    for (GemmW* g : {&vconv_, &pconv_, &vfc1_, &pfc_, &dense1_, &dense2_}) {
        g->w.free_();
        g->b.free_();
    }
    vfc2_w_.free_();
    fused_w_.free_();
    fused_b_.free_();
    fused_s_.free_();
    small_w_.free_();
    small_b_.free_();
    trace_.free_();
    flush_.free_();
}

// Weight layouts.
//  bf16: every contraction is D[rows x N] = A[rows x K] * W[N x K]^T with K-major bf16 operands, so each weight is
//        stored as [N_pad][K_pad] bf16 (+ f32 bias[N_pad]).  conv3x3: K index = tap * Cin_pad + c (tap = ky*3+kx);
//        FC: K index = cell * C_pad + c, i.e. the NCHW flatten order of net_utils.py:70,80 permuted to the NHWC order
//        the head convs write.
//  fp32 check mode: the blob's PyTorch layouts, untouched.
void Engine::upload_weights(const Blob& blob) {
    const uint32_t s2 = d_.s2();
    const float* D = blob.data.data();
    if (simple_) {
        // SimpleTwoHeadedModel: three dense layers over the NCHW-flattened planes (net_utils.py:112-121).  bf16: [N_pad][K_pad]
        // K-major like every other contraction here, K index = the flatten index itself; fp32 check mode: PyTorch layouts.
        const uint32_t nf = d_.features();
        auto dense = [&](GemmW& g, size_t w_off, size_t b_off, uint32_t n_out) {
            if (precision_ == CATTUS_B200_PRECISION_FP32_CHECK) {
                upload(g.w, std::vector<float>(D + w_off, D + w_off + static_cast<size_t>(n_out) * nf));
                upload(g.b, std::vector<float>(D + b_off, D + b_off + n_out));
                return;
            }
            if (n_out <= 128) {
                g.n_umma = round_up(n_out, 16);
                g.n_tiles = 1;
            } else {
                g.n_umma = 128;
                g.n_tiles = ceil_div(n_out, 128);
            }
            const uint32_t np = g.n_umma * g.n_tiles;
            g.k_pad = round_up(nf, 64);
            std::vector<float> w(static_cast<size_t>(np) * g.k_pad, 0.0f), b(np, 0.0f);
            for (uint32_t o = 0; o < n_out; ++o) {
                b[o] = D[b_off + o];
                for (uint32_t k = 0; k < nf; ++k) w[static_cast<size_t>(o) * g.k_pad + k] = D[w_off + static_cast<size_t>(o) * nf + k];
            }
            upload(g.w, to_bf16(tile_b(w, g)));
            upload(g.b, b);
        };
        dense(dense1_, blob.d1_w, blob.d1_b, nf);
        dense(dense2_, blob.d2_w, blob.d2_b, nf);
        dense(pfc_, blob.pfc_w, blob.pfc_b, d_.moves);
        upload(vfc2_w_, std::vector<float>(D + blob.vfc2_w, D + blob.vfc2_w + nf));
        vfc2_b_ = D[blob.vfc2_b];
        return;
    }
    if (precision_ == CATTUS_B200_PRECISION_FP32_CHECK) {
        auto up = [&](GemmW& g, size_t w, size_t wn, size_t b, size_t bn) {
            upload(g.w, std::vector<float>(D + w, D + w + wn));
            upload(g.b, std::vector<float>(D + b, D + b + bn));
        };
        auto upc = [&](GemmW& g, const Blob::Conv& c) { up(g, c.w, static_cast<size_t>(c.co) * c.ci * c.k * c.k, c.b, c.co); };
        convs_.resize(1 + blob.block_conv.size());
        upc(convs_[0], blob.stem);
        for (size_t i = 0; i < blob.block_conv.size(); ++i) upc(convs_[1 + i], blob.block_conv[i]);
        upc(vconv_, blob.vconv);
        upc(pconv_, blob.pconv);
        up(vfc1_, blob.vfc1_w, static_cast<size_t>(d_.hidden) * d_.vh * s2, blob.vfc1_b, d_.hidden);
        up(pfc_, blob.pfc_w, static_cast<size_t>(d_.moves) * d_.ph * s2, blob.pfc_b, d_.moves);
        upload(vfc2_w_, std::vector<float>(D + blob.vfc2_w, D + blob.vfc2_w + d_.hidden));
        vfc2_b_ = D[blob.vfc2_b];
        return;
    }
    auto n_split = [](uint32_t n, uint32_t& n_umma, uint32_t& n_tiles) {
        if (n <= 128) {
            n_umma = round_up(n, 16);
            n_tiles = 1;
        } else {
            n_umma = 128;
            n_tiles = ceil_div(n, 128);
        }
    };
    auto conv3 = [&](GemmW& g, const Blob::Conv& c, uint32_t ci_pad) {
        n_split(c.co, g.n_umma, g.n_tiles);
        const uint32_t np = g.n_umma * g.n_tiles;
        g.k_pad = 9 * ci_pad;
        std::vector<float> w(static_cast<size_t>(np) * g.k_pad, 0.0f), b(np, 0.0f);
        for (uint32_t o = 0; o < c.co; ++o) {
            b[o] = D[c.b + o];
            for (uint32_t i = 0; i < c.ci; ++i)
                for (uint32_t t = 0; t < 9; ++t) w[static_cast<size_t>(o) * g.k_pad + t * ci_pad + i] = D[c.w + (static_cast<size_t>(o) * c.ci + i) * 9 + t];
        }
        upload(g.w, to_bf16(tile_b(w, g)));
        upload(g.b, b);
    };
    auto conv1 = [&](GemmW& g, const Blob::Conv& c, uint32_t co_pad) {
        g.n_umma = co_pad;
        g.n_tiles = 1;
        g.k_pad = ca_;
        std::vector<float> w(static_cast<size_t>(co_pad) * ca_, 0.0f), b(co_pad, 0.0f);
        for (uint32_t o = 0; o < c.co; ++o) {
            b[o] = D[c.b + o];
            for (uint32_t i = 0; i < c.ci; ++i) w[static_cast<size_t>(o) * ca_ + i] = D[c.w + static_cast<size_t>(o) * c.ci + i];
        }
        upload(g.w, to_bf16(tile_b(w, g)));
        upload(g.b, b);
    };
    auto fc = [&](GemmW& g, size_t w_off, size_t b_off, uint32_t n_out, uint32_t ch, uint32_t ch_pad) {
        n_split(n_out, g.n_umma, g.n_tiles);
        const uint32_t np = g.n_umma * g.n_tiles;
        g.k_pad = round_up(s2 * ch_pad, 64);
        std::vector<float> w(static_cast<size_t>(np) * g.k_pad, 0.0f), b(np, 0.0f);
        for (uint32_t o = 0; o < n_out; ++o) {
            b[o] = D[b_off + o];
            for (uint32_t c = 0; c < ch; ++c)
                for (uint32_t cell = 0; cell < s2; ++cell)
                    w[static_cast<size_t>(o) * g.k_pad + cell * ch_pad + c] = D[w_off + static_cast<size_t>(o) * ch * s2 + c * s2 + cell];
        }
        upload(g.w, to_bf16(tile_b(w, g)));
        upload(g.b, b);
    };
    convs_.resize(1 + blob.block_conv.size());
    conv3(convs_[0], blob.stem, cin_pad_);
    for (size_t i = 0; i < blob.block_conv.size(); ++i) conv3(convs_[1 + i], blob.block_conv[i], ca_);
    if (fused_trunk_) {
        // trunk_fused.cuh weight image: for each layer, each k-chunk (16 input channels bf16, 32 e4m3), each CTA rank (= half of
        // the output channels) one block [tap 9][k-half 2][oc F / 2][16 bytes of ic] (8 bf16 / 16 e4m3 channels), streamed as one
        // TMA stage (F <= 128) or three (F = 256: 3 taps each).  Stem input channels padded to 32.  Last block per rank: the two
        // head convs, 8 k-chunks per stage.
        // FP8: every output channel of every conv (stem, block convs, head convs) is quantised on its own: amax_oc = max |w_oc|,
        // q = e4m3_rn_satfinite(w * (448 / amax_oc)), dequantisation factor d_oc = amax_oc / 448 (1 for an all-zero channel),
        // applied in the kernel's epilogue.  oracle/fp8.py: convnet_forward_fp8 does the same.
        const uint32_t layers = 1 + static_cast<uint32_t>(blob.block_conv.size());
        const uint32_t F = d_.f, ec = fp8_ ? 16 : 8, kcn = F / (2 * ec), stem_kc = 32 / (2 * ec), npc = F / 2;
        const size_t block_elems = static_cast<size_t>(9) * 2 * npc * ec;                   // FtG<F, E>::kBlockBytes / sizeof(E)
        const size_t stage_elems = static_cast<size_t>(F <= 128 ? 9 : 3) * 2 * npc * ec;   // FtG<F, E>::kWStage / sizeof(E)
        const uint32_t head_stages = kcn > 8 ? kcn / 8 : 1, head_kc = kcn / head_stages;
        const size_t blocks = stem_kc + static_cast<size_t>(layers - 1) * kcn + 1;  // + one block for the two head convs
        std::vector<float> img(blocks * 2 * block_elems, 0.0f), bias(static_cast<size_t>(layers + 1) * F, 0.0f);
        std::vector<float> dq(bias.size(), 1.0f), qs(bias.size(), 1.0f);  // FP8: d_oc and 448 / amax_oc per [layer][oc]
        auto set_scale = [&](size_t row, float amax) {
            if (fp8_ && amax > 0.0f) {
                qs[row] = 448.0f / amax;
                dq[row] = amax / 448.0f;
            }
        };
        for (uint32_t l = 0; l < layers; ++l) {
            const Blob::Conv& c = l == 0 ? blob.stem : blob.block_conv[l - 1];
            const uint32_t nkc = l == 0 ? stem_kc : kcn;
            const size_t base = l == 0 ? 0 : stem_kc + static_cast<size_t>(l - 1) * kcn;
            for (uint32_t o = 0; o < F; ++o) {
                bias[l * F + o] = D[c.b + o];
                float amax = 0.0f;
                for (size_t i = 0; i < static_cast<size_t>(c.ci) * 9; ++i) amax = std::max(amax, std::fabs(D[c.w + static_cast<size_t>(o) * c.ci * 9 + i]));
                set_scale(static_cast<size_t>(l) * F + o, amax);
            }
            for (uint32_t kc = 0; kc < nkc; ++kc)
                for (uint32_t rk = 0; rk < 2; ++rk) {
                    float* blk = img.data() + ((base + kc) * 2 + rk) * block_elems;
                    for (uint32_t tap = 0; tap < 9; ++tap)
                        for (uint32_t kh = 0; kh < 2; ++kh)
                            for (uint32_t n = 0; n < npc; ++n)
                                for (uint32_t e2 = 0; e2 < ec; ++e2) {
                                    const uint32_t ic = kc * 2 * ec + kh * ec + e2, oc = rk * npc + n;
                                    if (ic < c.ci)
                                        blk[((tap * 2 + kh) * npc + n) * ec + e2] = D[c.w + (static_cast<size_t>(oc) * c.ci + ic) * 9 + tap] * qs[static_cast<size_t>(l) * F + oc];
                                }
                }
        }
        {
            // head stages: [k-chunk][k-half 2][oc (vhp + php) / 2][16 bytes of ic] per CTA rank; channel list = value | policy
            const uint32_t nh = vhp_ + php_, half = nh / 2;
            const size_t base = stem_kc + static_cast<size_t>(layers - 1) * kcn;
            const size_t hrow = static_cast<size_t>(layers) * F;
            auto head_w = [&](uint32_t ch, uint32_t ic) -> float {
                if (ch < vhp_) return ch < d_.vh ? D[blob.vconv.w + static_cast<size_t>(ch) * F + ic] : 0.0f;
                const uint32_t pc = ch - vhp_;
                return pc < d_.ph ? D[blob.pconv.w + static_cast<size_t>(pc) * F + ic] : 0.0f;
            };
            for (uint32_t ch = 0; ch < nh; ++ch) {
                float amax = 0.0f;
                for (uint32_t ic = 0; ic < F; ++ic) amax = std::max(amax, std::fabs(head_w(ch, ic)));
                set_scale(hrow + ch, amax);
            }
            for (uint32_t rk = 0; rk < 2; ++rk) {
                float* blk = img.data() + (base * 2 + rk) * block_elems;
                for (uint32_t kc = 0; kc < kcn; ++kc) {
                    float* st = blk + (kc / head_kc) * stage_elems;
                    const uint32_t k8 = kc % head_kc;
                    for (uint32_t kh = 0; kh < 2; ++kh)
                        for (uint32_t n = 0; n < half; ++n)
                            for (uint32_t e2 = 0; e2 < ec; ++e2)
                                st[((k8 * 2 + kh) * half + n) * ec + e2] = head_w(rk * half + n, kc * 2 * ec + kh * ec + e2) * qs[hrow + rk * half + n];
                }
            }
            for (uint32_t o = 0; o < d_.vh; ++o) bias[hrow + o] = D[blob.vconv.b + o];
            for (uint32_t o = 0; o < d_.ph; ++o) bias[hrow + vhp_ + o] = D[blob.pconv.b + o];
        }
        if (fp8_) {
            std::vector<uint8_t> q(img.size());
            for (size_t i = 0; i < img.size(); ++i) q[i] = static_cast<uint8_t>(__nv_cvt_float_to_fp8(img[i], __NV_SATFINITE, __NV_E4M3));
            upload(fused_w_, q);
            upload(fused_s_, dq);
        } else {
            upload(fused_w_, to_bf16(img));
        }
        upload(fused_b_, bias);
    }
    if (small_trunk_) {
        // trunk_small.cuh weight image: per layer, per 16-channel k-chunk, per tap: [k-half 2][oc 16][ic 8] bf16 (512 B);
        // then the two head convs as one [k-half 2][oc vhp + php][ic 8] tile (value channels first).  Biases: [layers][16], [nh].
        const uint32_t layers = 1 + static_cast<uint32_t>(blob.block_conv.size());
        const uint32_t nh = vhp_ + php_;
        const size_t layer_elems = 9 * 256;
        std::vector<float> img((small_stem_kc_ + (layers - 1)) * layer_elems + 2 * nh * 8, 0.0f), bias(static_cast<size_t>(layers) * 16 + nh, 0.0f);
        size_t off = 0;
        for (uint32_t l = 0; l < layers; ++l) {
            const Blob::Conv& c = l == 0 ? blob.stem : blob.block_conv[l - 1];
            const uint32_t nkc = l == 0 ? small_stem_kc_ : 1;
            for (uint32_t o = 0; o < 16; ++o) bias[l * 16 + o] = D[c.b + o];
            for (uint32_t kc = 0; kc < nkc; ++kc)
                for (uint32_t tap = 0; tap < 9; ++tap)
                    for (uint32_t kh = 0; kh < 2; ++kh)
                        for (uint32_t o = 0; o < 16; ++o)
                            for (uint32_t e = 0; e < 8; ++e) {
                                const uint32_t ic = kc * 16 + kh * 8 + e;
                                if (ic < c.ci) img[off + ((kc * 9 + tap) * 2 + kh) * 128 + o * 8 + e] = D[c.w + (static_cast<size_t>(o) * c.ci + ic) * 9 + tap];
                            }
            off += nkc * layer_elems;
        }
        for (uint32_t kh = 0; kh < 2; ++kh)
            for (uint32_t e = 0; e < 8; ++e) {
                const uint32_t ic = kh * 8 + e;
                for (uint32_t o = 0; o < d_.vh; ++o) img[off + (kh * nh + o) * 8 + e] = D[blob.vconv.w + static_cast<size_t>(o) * 16 + ic];
                for (uint32_t o = 0; o < d_.ph; ++o) img[off + (kh * nh + vhp_ + o) * 8 + e] = D[blob.pconv.w + static_cast<size_t>(o) * 16 + ic];
            }
        for (uint32_t o = 0; o < d_.vh; ++o) bias[static_cast<size_t>(layers) * 16 + o] = D[blob.vconv.b + o];
        for (uint32_t o = 0; o < d_.ph; ++o) bias[static_cast<size_t>(layers) * 16 + vhp_ + o] = D[blob.pconv.b + o];
        upload(small_w_, to_bf16(img));
        upload(small_b_, bias);
    }
    conv1(vconv_, blob.vconv, vhp_);
    conv1(pconv_, blob.pconv, php_);
    fc(vfc1_, blob.vfc1_w, blob.vfc1_b, d_.hidden, d_.vh, vhp_);
    fc(pfc_, blob.pfc_w, blob.pfc_b, d_.moves, d_.ph, php_);
    upload(vfc2_w_, std::vector<float>(D + blob.vfc2_w, D + blob.vfc2_w + d_.hidden));
    vfc2_b_ = D[blob.vfc2_b];
}

void Engine::init_lane(Lane& l) {
    CB2_CUDA(cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking));
    CB2_CUDA(cudaEventCreateWithFlags(&l.done, cudaEventDisableTiming));
    const size_t in_bytes = kRecs0 + static_cast<size_t>(max_batch_) * rec_.rec_bytes;
    CB2_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&l.h_in), in_bytes, cudaHostAllocDefault));
    std::memset(l.h_in, 0, in_bytes);
    CB2_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&l.h_values), sizeof(float) * max_batch_, cudaHostAllocMapped));
    CB2_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&l.h_probs), sizeof(float) * max_batch_ * d_.moves, cudaHostAllocMapped));
    CB2_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&l.zc_values), l.h_values, 0));
    CB2_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&l.zc_probs), l.h_probs, 0));
    l.d_in.alloc(in_bytes);
    l.d_values.alloc(sizeof(float) * max_batch_);
    l.d_probs.alloc(sizeof(float) * max_batch_ * d_.moves);
    const uint32_t s2 = d_.s2();
    l.d_dense.alloc(sizeof(float) * max_batch_ * d_.c_in * s2);
    if (simple_) {
        // activations are [max_batch][K_pad] rows (bf16) / [max_batch][n] (fp32); columns beyond a layer's width stay zero
        const size_t nf = d_.features(), kp = round_up(static_cast<uint32_t>(nf), 64);
        const bool f32 = precision_ == CATTUS_B200_PRECISION_FP32_CHECK;
        const size_t row_bytes = f32 ? nf * 4 : std::max<size_t>(kp, dense1_.n_umma * dense1_.n_tiles) * 2;
        l.d_x.alloc(row_bytes * max_batch_);
        l.d_act[0].alloc(row_bytes * max_batch_);
        l.d_act[1].alloc(row_bytes * max_batch_);
        l.d_logits.alloc(sizeof(float) * max_batch_ * (f32 ? d_.moves : pfc_.n_umma * pfc_.n_tiles));
        return;
    }
    l.d_hidden.alloc(sizeof(float) * max_batch_ * d_.hidden);
    if (precision_ == CATTUS_B200_PRECISION_FP32_CHECK) {
        l.d_x.alloc(sizeof(float) * max_batch_ * d_.c_in * s2);
        for (auto& a : l.d_act) a.alloc(sizeof(float) * max_batch_ * d_.f * s2);
        l.d_hv.alloc(sizeof(float) * max_batch_ * d_.vh * s2);
        l.d_hp.alloc(sizeof(float) * max_batch_ * d_.ph * s2);
        l.d_logits.alloc(sizeof(float) * max_batch_ * d_.moves);
    } else {
        const size_t rows = static_cast<size_t>(round_up(max_batch_, nb_)) * s2;
        l.d_x.alloc(rows * cin_pad_ * 2);
        for (auto& a : l.d_act) a.alloc(rows * ca_ * 2);
        l.d_hv.alloc(rows * vhp_ * 2);
        l.d_hp.alloc(rows * php_ * 2);
        l.d_logits.alloc(sizeof(float) * max_batch_ * pfc_.n_umma * pfc_.n_tiles);
    }
}

uint32_t Engine::bucket_for(uint32_t n) const {
    uint32_t b = 1;
    while (b < n) b <<= 1;
    return std::min(b, max_batch_);
}

// ------------------------------------------------------------------------------------------------ tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

CUtensorMap Engine::make_map_2d(const void* base, uint64_t inner, uint64_t rows, uint64_t row_stride_bytes, uint32_t box_rows) {
    CUtensorMap m;
    cuuint64_t gdim[2] = {inner, rows};
    cuuint64_t gstr[1] = {row_stride_bytes};
    cuuint32_t box[2] = {64, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = reinterpret_cast<EncodeTiledFn>(encode_tiled_)(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr,
                                                                box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                                                CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) throw Error(CATTUS_B200_ECUDA, "cuTensorMapEncodeTiled(2d) failed with " + std::to_string(static_cast<int>(r)));
    return m;
}


// NHWC activations [boards][S][S][channels]; box = {64 channels, S, S, nb boards}.  Out-of-bounds halo -> zeros.
CUtensorMap Engine::make_map_conv(const void* base, uint32_t channels, uint32_t boards, uint32_t nb) {
    CUtensorMap m;
    const uint64_t s = d_.s;
    cuuint64_t gdim[4] = {channels, s, s, boards};
    cuuint64_t gstr[3] = {channels * 2ull, s * channels * 2ull, s * s * channels * 2ull};
    cuuint32_t box[4] = {64, static_cast<cuuint32_t>(s), static_cast<cuuint32_t>(s), nb};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = reinterpret_cast<EncodeTiledFn>(encode_tiled_)(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), gdim, gstr,
                                                                box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                                                CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) throw Error(CATTUS_B200_ECUDA, "cuTensorMapEncodeTiled(4d) failed with " + std::to_string(static_cast<int>(r)));
    return m;
}

// Ring of the GEMM kernel: the deep form (3 slots of two k-blocks = 6 tile pairs, one CTA per SM) for the smallest batches
// (<= 64 rows) of GEMMs with a long k-loop (the chess head FCs, 32 k-blocks: B = 1 ... 64 graph -2 to -4 us); 3 slots of
// one k-block and two CTAs per SM otherwise.
// Short k-loops gain nothing from the depth and the 197 KB launch costs the hex5 graph 2-4 us; larger small batches
// usually come from many lanes at once (trainer-sized jobs with speculative rows: ~100 rows per batch on 16 streams),
// where CTAs that each take a whole SM cost 12 % of the job's throughput (1.24 M -> 1.09 M sims/s), more than the 2-4 us
// they save a lone batch.  A/B knob: CATTUS_B200_TC_NO_DEEP.  (Round 1 measured no gain from the deep ring at all: the
// k-loop was then paced by the single-lane issue loops, not by the loads -- see tc_gemm.cuh.)
int Engine::tc_stages_for(uint32_t ctas, int num_kb, uint32_t rows) const {
    static const bool no_deep = std::getenv("CATTUS_B200_TC_NO_DEEP") != nullptr;
    return !no_deep && ctas <= static_cast<uint32_t>(sm_count_) && num_kb >= 16 && num_kb % 2 == 0 && rows <= 64 ? kTcStagesDeep : kTcStages;
}

// Launch with programmatic stream serialization: the kernel may be staged while its predecessor on the stream still runs
// (ptx.cuh: grid_dep_wait / grid_dep_launch).  Captured into the bucket graphs as a programmatic dependency edge.
template <class... P, class... Args>
static void launch_pdl(void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    static const bool off = std::getenv("CATTUS_B200_NO_PDL") != nullptr;  // A/B knob
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = off ? 0 : 1;
    CB2_CUDA(cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...));
}

Op Engine::make_tc_op(int stage, const char* name, const TcGemmParams& p, uint32_t m_tiles, uint32_t n_tiles) {
    Op op;
    op.stage = stage;
    op.name = name;
    const dim3 grid(m_tiles, n_tiles);
    TcGemmParams q = p;
    const int stages = tc_stages_for(m_tiles * n_tiles, p.num_kb, p.mode == 0 ? static_cast<uint32_t>(p.m_valid) : 0xFFFFFFFFu);
    q.fault = (desc_.flags & 2u) && stage == 2 ? 1 : 0;
    const int smem_bytes = tc_smem_bytes(stages);
    if (stages == kTcStagesDeep)
        op.launch = [q, grid, smem_bytes](cudaStream_t st) { tc_gemm_kernel<2><<<grid, kTcThreads, smem_bytes, st>>>(q); };
    else
        op.launch = [q, grid, smem_bytes](cudaStream_t st) { tc_gemm_kernel<1><<<grid, kTcThreads, smem_bytes, st>>>(q); };
    return op;
}

// ------------------------------------------------------------------------------------------------ op lists
static inline int grid_for(long long work_items, int threads, int sm_count) {
    long long blocks = (work_items + threads - 1) / threads;
    const long long cap = static_cast<long long>(sm_count) * 16;
    return static_cast<int>(std::max<long long>(1, std::min(blocks, cap)));
}

std::vector<Op>& Engine::ops_for(Lane& lane, uint32_t bucket, bool dense_input) {
    const uint32_t key = bucket | (dense_input ? 0x80000000u : 0u) | (lane.device_out ? 0x40000000u : 0u);
    auto it = lane.ops.find(key);
    if (it != lane.ops.end()) return it->second;
    std::vector<Op> ops;
    if (simple_)
        build_ops_simple(lane, bucket, ops, dense_input);
    else if (precision_ == CATTUS_B200_PRECISION_FP32_CHECK)
        build_ops_fp32(lane, bucket, ops, dense_input);
    else
        build_ops_bf16(lane, bucket, ops, dense_input);
    return lane.ops.emplace(key, std::move(ops)).first->second;
}

void Engine::add_tail_ops(Lane& lane, uint32_t bucket, std::vector<Op>& ops, bool dense_input, bool value_tail, bool policy_tail) {
    const uint8_t* recs = lane.d_in.as<uint8_t>() + kRecs0;
    const uint32_t* n_ptr = lane.d_in.as<uint32_t>();
    const RecLayout L = rec_;
    const int ld_logits = precision_ == CATTUS_B200_PRECISION_FP32_CHECK ? static_cast<int>(d_.moves) : static_cast<int>(pfc_.n_umma * pfc_.n_tiles);
    if (value_tail) {
        Op op;
        op.stage = 3;
        op.name = "value_tail";
        const float* hidden = lane.d_hidden.as<float>();
        const float* w2 = vfc2_w_.as<float>();
        const float b2 = vfc2_b_;
        float* values = zero_copy_out(lane, bucket, dense_input) ? lane.zc_values : lane.d_values.as<float>();
        const int blocks = static_cast<int>(ceil_div(bucket * 32, 256));
        op.launch = [=](cudaStream_t st) { value_tail_kernel<<<blocks, 256, 0, st>>>(hidden, 128, w2, b2, n_ptr, values); };
        ops.push_back(op);
    }
    if (dense_input || !policy_tail) return;  // run_dense returns raw logits (Model::run semantics)
    {
        Op op;
        op.stage = 3;
        op.name = "policy_tail";
        const float* logits = lane.d_logits.as<float>();
        float* probs = zero_copy_out(lane, bucket, dense_input) ? lane.zc_probs : lane.d_probs.as<float>();
        const int blocks = static_cast<int>(ceil_div(bucket * 32, 256));
        op.launch = [=](cudaStream_t st) { policy_tail_kernel<<<blocks, 256, 0, st>>>(logits, ld_logits, recs, L, n_ptr, probs); };
        ops.push_back(op);
    }
}

// SimpleTwoHeadedModel.forward (net_utils.py:112-121): flatten -> dense1 + ReLU -> dense2 + ReLU -> {policy, tanh(value)}.
// bf16: three tcgen05 GEMMs (tc_gemm.cuh) over [positions][K_pad] rows + a warp-per-position value dot product;
// fp32 check mode: the CUDA-core loops.  The policy tail is the standalone clamp + mask + softmax kernel.
void Engine::build_ops_simple(Lane& lane, uint32_t bucket, std::vector<Op>& ops, bool dense_input) {
    const int n = static_cast<int>(bucket);
    const int nf = static_cast<int>(d_.features());
    const uint8_t* recs = lane.d_in.as<uint8_t>() + kRecs0;
    const uint32_t* n_ptr = lane.d_in.as<uint32_t>();
    const RecLayout L = rec_;
    const int sm = sm_count_;
    float* values = zero_copy_out(lane, bucket, dense_input) ? lane.zc_values : lane.d_values.as<float>();
    const float* w2 = vfc2_w_.as<float>();
    const float b2 = vfc2_b_;
    const int vblocks = static_cast<int>(ceil_div(bucket * 32, 256));
    if (precision_ == CATTUS_B200_PRECISION_FP32_CHECK) {
        const float* x = dense_input ? lane.d_dense.as<float>() : lane.d_x.as<float>();
        if (!dense_input) {
            Op op;
            op.stage = 0;
            op.name = "encode_nchw_f32";
            float* out = lane.d_x.as<float>();
            const int blocks = grid_for(static_cast<long long>(n) * nf, 256, sm);
            op.launch = [=](cudaStream_t st) { encode_nchw_f32_kernel<<<blocks, 256, 0, st>>>(recs, L, n_ptr, n, out); };
            ops.push_back(op);
        }
        auto fc = [&](int stage, const char* name, const float* in, const GemmW& g, float* out, int no, int relu) {
            Op op;
            op.stage = stage;
            op.name = name;
            const float* w = g.w.as<float>();
            const float* b = g.b.as<float>();
            const int blocks = grid_for(static_cast<long long>(n) * no * 32, 256, sm);
            op.launch = [=](cudaStream_t st) { fc_f32_kernel<<<blocks, 256, 0, st>>>(in, w, b, out, n, nf, no, no, relu); };
            ops.push_back(op);
        };
        float* a0 = lane.d_act[0].as<float>();
        float* a1 = lane.d_act[1].as<float>();
        fc(1, "dense1", x, dense1_, a0, nf, 1);
        fc(1, "dense2", a0, dense2_, a1, nf, 1);
        {
            Op op;
            op.stage = 2;
            op.name = "value_dot_tanh";
            op.launch = [=](cudaStream_t st) { dot_tanh_kernel<float><<<vblocks, 256, 0, st>>>(a1, nf, nf, w2, b2, n_ptr, n, values); };
            ops.push_back(op);
        }
        fc(2, "policy", a1, pfc_, lane.d_logits.as<float>(), static_cast<int>(d_.moves), 0);
    } else {
        const int kp = static_cast<int>(dense1_.k_pad);
        const int ld = static_cast<int>(std::max<uint32_t>(dense1_.k_pad, dense1_.n_umma * dense1_.n_tiles));
        __nv_bfloat16* x = lane.d_x.as<__nv_bfloat16>();
        {
            Op op;
            op.stage = 0;
            const int blocks = grid_for(static_cast<long long>(n) * (kp / 8), 256, sm);
            if (dense_input) {
                op.name = "nchw_f32_to_flat_bf16";
                const float* in = lane.d_dense.as<float>();
                op.launch = [=](cudaStream_t st) { nchw_f32_to_flat_bf16_kernel<<<blocks, 256, 0, st>>>(in, n, nf, kp, ld, x); };
            } else {
                op.name = "encode_flat_bf16";
                op.launch = [=](cudaStream_t st) { encode_flat_bf16_kernel<<<blocks, 256, 0, st>>>(recs, L, n_ptr, n, nf, kp, ld, x); };
            }
            ops.push_back(op);
        }
        auto gemm = [&](int stage, const char* name, const void* a, const GemmW& g, void* out, uint32_t ld_out, bool out_f32, bool relu) {
            TcGemmParams p;
            std::memset(&p, 0, sizeof(p));
            p.err = d_err_;
            p.s2 = static_cast<int>(d_.s2());
            p.nb = 1;
            p.tma_a = make_map_2d(a, static_cast<uint64_t>(nf), bucket, static_cast<uint64_t>(ld) * 2, std::min(128u, bucket));
            p.b_img = g.w.as<uint8_t>();
            p.bias = g.b.as<float>();
            p.out = out;
            p.mode = 0;
            p.kh = 1;
            p.num_kb = static_cast<int>(g.k_pad / 64);
            p.n_umma = static_cast<int>(g.n_umma);
            p.n_store = static_cast<int>(g.n_umma);
            p.m_valid = static_cast<int>(bucket);
            p.rows_per_tile = 128;
            p.ld_out = static_cast<int>(ld_out);
            p.out_f32 = out_f32 ? 1 : 0;
            p.relu = relu ? 1 : 0;
            p.tx_bytes = std::min(128u, bucket) * 128 + g.n_umma * 128;
            ops.push_back(make_tc_op(stage, name, p, ceil_div(bucket, 128), g.n_tiles));
        };
        __nv_bfloat16* a0 = lane.d_act[0].as<__nv_bfloat16>();
        __nv_bfloat16* a1 = lane.d_act[1].as<__nv_bfloat16>();
        gemm(1, "dense1", x, dense1_, a0, static_cast<uint32_t>(ld), false, true);
        gemm(1, "dense2", a0, dense2_, a1, static_cast<uint32_t>(ld), false, true);
        {
            Op op;
            op.stage = 2;
            op.name = "value_dot_tanh";
            op.launch = [=](cudaStream_t st) { dot_tanh_kernel<__nv_bfloat16><<<vblocks, 256, 0, st>>>(a1, ld, nf, w2, b2, n_ptr, n, values); };
            ops.push_back(op);
        }
        gemm(2, "policy", a1, pfc_, lane.d_logits.p, pfc_.n_umma * pfc_.n_tiles, true, false);
    }
    if (dense_input) return;  // run_dense returns raw logits (Model::run semantics)
    Op op;
    op.stage = 3;
    op.name = "policy_tail";
    const float* logits = lane.d_logits.as<float>();
    const int ld_logits = precision_ == CATTUS_B200_PRECISION_FP32_CHECK ? static_cast<int>(d_.moves) : static_cast<int>(pfc_.n_umma * pfc_.n_tiles);
    float* probs = zero_copy_out(lane, bucket, dense_input) ? lane.zc_probs : lane.d_probs.as<float>();
    const int blocks = static_cast<int>(ceil_div(bucket * 32, 256));
    op.launch = [=](cudaStream_t st) { policy_tail_kernel<<<blocks, 256, 0, st>>>(logits, ld_logits, recs, L, n_ptr, probs); };
    ops.push_back(op);
}

void Engine::build_ops_fp32(Lane& lane, uint32_t bucket, std::vector<Op>& ops, bool dense_input) {
    const int s = static_cast<int>(d_.s), s2 = static_cast<int>(d_.s2());
    const int n = static_cast<int>(bucket);
    const uint8_t* recs = lane.d_in.as<uint8_t>() + kRecs0;
    const uint32_t* n_ptr = lane.d_in.as<uint32_t>();
    const RecLayout L = rec_;
    const int sm = sm_count_;
    const float* x = dense_input ? lane.d_dense.as<float>() : lane.d_x.as<float>();
    if (!dense_input) {
        Op op;
        op.stage = 0;
        op.name = "encode_nchw_f32";
        float* out = lane.d_x.as<float>();
        const long long total = static_cast<long long>(n) * d_.c_in * s2;
        const int blocks = grid_for(total, 256, sm);
        op.launch = [=](cudaStream_t st) { encode_nchw_f32_kernel<<<blocks, 256, 0, st>>>(recs, L, n_ptr, n, out); };
        ops.push_back(op);
    }
    auto conv = [&](int stage, const char* name, const float* in, const GemmW& g, const float* resid, float* out, int ci, int co, int ks, int relu) {
        Op op;
        op.stage = stage;
        op.name = name;
        const float* w = g.w.as<float>();
        const float* b = g.b.as<float>();
        const long long total = static_cast<long long>(n) * co * s2;
        const int blocks = grid_for(total, 128, sm);
        op.launch = [=](cudaStream_t st) { conv_f32_kernel<<<blocks, 128, 0, st>>>(in, w, b, resid, out, n, ci, co, s, ks, relu); };
        ops.push_back(op);
    };
    auto fc = [&](const char* name, const float* in, const GemmW& g, float* out, int k, int no, int ld, int relu) {
        Op op;
        op.stage = 2;
        op.name = name;
        const float* w = g.w.as<float>();
        const float* b = g.b.as<float>();
        const long long total = static_cast<long long>(n) * no * 32;
        const int blocks = grid_for(total, 256, sm);
        op.launch = [=](cudaStream_t st) { fc_f32_kernel<<<blocks, 256, 0, st>>>(in, w, b, out, n, k, no, ld, relu); };
        ops.push_back(op);
    };
    float* act[3] = {lane.d_act[0].as<float>(), lane.d_act[1].as<float>(), lane.d_act[2].as<float>()};
    const int F = static_cast<int>(d_.f);
    conv(1, "stem", x, convs_[0], nullptr, act[0], static_cast<int>(d_.c_in), F, 3, 1);
    int cur = 0;
    for (uint32_t i = 0; i < d_.r; ++i) {
        const int h = (cur + 1) % 3, o = (cur + 2) % 3;
        conv(1, "block_conv1", act[cur], convs_[1 + 2 * i], nullptr, act[h], F, F, 3, 1);
        conv(1, "block_conv2", act[h], convs_[2 + 2 * i], act[cur], act[o], F, F, 3, 1);
        cur = o;
    }
    conv(2, "value_conv", act[cur], vconv_, nullptr, lane.d_hv.as<float>(), F, static_cast<int>(d_.vh), 1, 1);
    conv(2, "policy_conv", act[cur], pconv_, nullptr, lane.d_hp.as<float>(), F, static_cast<int>(d_.ph), 1, 1);
    fc("value_fc1", lane.d_hv.as<float>(), vfc1_, lane.d_hidden.as<float>(), static_cast<int>(d_.vh) * s2, 128, 128, 1);
    fc("policy_fc", lane.d_hp.as<float>(), pfc_, lane.d_logits.as<float>(), static_cast<int>(d_.ph) * s2, static_cast<int>(d_.moves),
       static_cast<int>(d_.moves), 0);
    add_tail_ops(lane, bucket, ops, dense_input, true, true);
}

void Engine::build_ops_bf16(Lane& lane, uint32_t bucket, std::vector<Op>& ops, bool dense_input) {
    const uint32_t s2 = d_.s2();
    const uint32_t tiles = ceil_div(bucket, nb_);
    const uint32_t boards = tiles * nb_;
    const uint32_t rows_total = boards * s2;
    const uint8_t* recs = lane.d_in.as<uint8_t>() + kRecs0;
    const uint32_t* n_ptr = lane.d_in.as<uint32_t>();
    const RecLayout L = rec_;
    const int sm = sm_count_;
    __nv_bfloat16* x = lane.d_x.as<__nv_bfloat16>();
    const bool fused = fused_trunk_ && !dense_input;
    const bool small = small_trunk_ && !dense_input;
    if (!fused && !small) {
        Op op;
        op.stage = 0;
        const int blocks = grid_for(static_cast<long long>(rows_total) * (cin_pad_ / 8), 256, sm);
        const int rt = static_cast<int>(rows_total);
        if (dense_input) {
            op.name = "nchw_f32_to_nhwc_bf16";
            const float* in = lane.d_dense.as<float>();
            const int n = static_cast<int>(bucket), ci = static_cast<int>(d_.c_in), is2 = static_cast<int>(s2);
            const int blocks64 = grid_for(static_cast<long long>(rows_total) * 64, 256, sm);
            if (cin_pad_ != 64) throw Error(CATTUS_B200_EINVAL, "planes > 64 not supported");
            op.launch = [=](cudaStream_t st) { nchw_f32_to_nhwc_bf16_kernel<<<blocks64, 256, 0, st>>>(in, n, ci, is2, rt, x); };
        } else {
            op.name = "encode_nhwc_bf16";
            op.launch = [=](cudaStream_t st) { encode_nhwc_bf16_kernel<<<blocks, 256, 0, st>>>(recs, L, n_ptr, rt, x); };
        }
        ops.push_back(op);
    }
    auto base_params = [&]() {
        TcGemmParams p;
        std::memset(&p, 0, sizeof(p));
        p.err = d_err_;
        p.s2 = static_cast<int>(s2);
        p.nb = static_cast<int>(nb_);
        p.n_ptr = n_ptr;  // M tiles of nothing but padding positions return at once
        return p;
    };
    // 3x3 conv: A = NHWC activations through the 4-D halo map, B = [Np][9*Cpad]
    auto conv3 = [&](const char* name, const __nv_bfloat16* in, uint32_t cpad, const GemmW& g, const __nv_bfloat16* resid, __nv_bfloat16* out) {
        TcGemmParams p = base_params();
        p.tma_a = make_map_conv(in, cpad, boards, nb_);
        p.b_img = g.w.as<uint8_t>();
        p.bias = g.b.as<float>();
        p.resid = resid;
        p.out = out;
        p.mode = 1;
        p.kh = static_cast<int>(cpad / 64);
        p.num_kb = 9 * p.kh;
        p.n_umma = static_cast<int>(g.n_umma);
        p.n_store = static_cast<int>(g.n_umma);
        p.m_valid = static_cast<int>(boards);
        p.rows_per_tile = static_cast<int>(nb_ * s2);
        p.ld_out = static_cast<int>(ca_);
        p.out_f32 = 0;
        p.relu = 1;
        p.tx_bytes = nb_ * s2 * 128 + g.n_umma * 128;
        ops.push_back(make_tc_op(1, name, p, tiles, g.n_tiles));
    };
    TcGemmParams last_tc;  // parameters of the most recent gemm() op (the fused-tail variants are derived from them)
    std::memset(&last_tc, 0, sizeof(last_tc));
    // plain GEMM: A = [rows][K] row-major bf16
    auto gemm = [&](int stage, const char* name, const void* a, uint64_t k_real, uint64_t rows, uint64_t row_stride_bytes, const GemmW& g,
                    void* out, uint32_t ld_out, bool out_f32, bool relu) {
        TcGemmParams p = base_params();
        const uint32_t a_rows = static_cast<uint32_t>(std::min<uint64_t>(128, rows));
        p.tma_a = make_map_2d(a, k_real, rows, row_stride_bytes, a_rows);
        p.b_img = g.w.as<uint8_t>();
        p.bias = g.b.as<float>();
        p.out = out;
        p.mode = 0;
        p.kh = 1;
        p.num_kb = static_cast<int>(g.k_pad / 64);
        p.n_umma = static_cast<int>(g.n_umma);
        p.n_store = static_cast<int>(g.n_umma);
        p.m_valid = static_cast<int>(rows);
        p.rows_per_tile = 128;
        p.ld_out = static_cast<int>(ld_out);
        p.out_f32 = out_f32 ? 1 : 0;
        p.relu = relu ? 1 : 0;
        p.tx_bytes = a_rows * 128 + g.n_umma * 128;
        last_tc = p;
        ops.push_back(make_tc_op(stage, name, p, ceil_div(static_cast<uint32_t>(rows), 128), g.n_tiles));
    };
    __nv_bfloat16* act[3] = {lane.d_act[0].as<__nv_bfloat16>(), lane.d_act[1].as<__nv_bfloat16>(), lane.d_act[2].as<__nv_bfloat16>()};
    int cur = 0;
    if (fused) {
        // encode + stem + all residual blocks in one persistent cluster launch (trunk_fused.cuh)
        TrunkFusedParams fp;
        std::memset(&fp, 0, sizeof(fp));
        const uint64_t w_rows = fused_w_.bytes / 256;
        {
            cuuint64_t gdim[2] = {256, w_rows};
            cuuint64_t gstr[1] = {256};
            using B = __nv_bfloat16;  // stage bytes are the same for both element types
            const int rows_per_stage = d_.f == 64 ? FtG<64, B>::kWRowsPerStage : d_.f == 128 ? FtG<128, B>::kWRowsPerStage : FtG<256, B>::kWRowsPerStage;
            cuuint32_t box[2] = {256, static_cast<cuuint32_t>(rows_per_stage)};
            cuuint32_t estr[2] = {1, 1};
            CUresult r = reinterpret_cast<EncodeTiledFn>(encode_tiled_)(&fp.tma_w, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, fused_w_.p, gdim, gstr, box, estr,
                                                                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                                                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) throw Error(CATTUS_B200_ECUDA, "cuTensorMapEncodeTiled(weights) failed with " + std::to_string(static_cast<int>(r)));
        }
        fp.recs = recs;
        fp.n_ptr = n_ptr;
        fp.bias = fused_b_.as<float>();
        fp.scale = fp8_ ? fused_s_.as<float>() : nullptr;
        fp.out_v = lane.d_hv.as<__nv_bfloat16>();
        fp.out_p = lane.d_hp.as<__nv_bfloat16>();
        fp.vhp = static_cast<int>(vhp_);
        fp.php = static_cast<int>(php_);
        fp.err = d_err_;
        fp.rec_bytes = rec_.rec_bytes;
        fp.planes = static_cast<int>(d_.c_in);
        fp.layers = 1 + 2 * static_cast<int>(d_.r);
        fp.dbg = nullptr;
        if (std::getenv("CATTUS_B200_TRACE_TRUNK")) {  // diagnostic: per-layer clock64 trace of pair 0, printed by time_stage
            if (trace_.p == nullptr) trace_.alloc(512 * sizeof(unsigned long long));
            fp.dbg = trace_.as<unsigned long long>();
        }
        // small batches: one tile per CTA (4 boards per pair) while that still fits one wave -- half the MMAs per round
        // (256 filters: one tile per CTA always -- two tiles' activations do not fit beside the weight ring)
        fp.tiles = (static_cast<int>(ceil_div(bucket, 4)) <= sm / 2 || d_.f == 256) ? 1 : 2;
        fp.num_rounds = static_cast<int>(ceil_div(bucket, 4u * static_cast<uint32_t>(fp.tiles)));
        const int pairs = std::min(sm / 2, fp.num_rounds);
        Op op;
        op.stage = 1;
        op.name = fp8_ ? "trunk_fused_fp8" : "trunk_fused";
        using B = __nv_bfloat16;
        using E8 = __nv_fp8_e4m3;
        if (d_.f == 64 && !fp8_)
            op.launch = [fp, pairs](cudaStream_t st) { trunk_fused_kernel<64, B><<<2 * pairs, kFtThreads, FtG<64, B>::kSmemBytes, st>>>(fp); };
        else if (d_.f == 128 && !fp8_)
            op.launch = [fp, pairs](cudaStream_t st) { trunk_fused_kernel<128, B><<<2 * pairs, kFtThreads, FtG<128, B>::kSmemBytes, st>>>(fp); };
        else if (!fp8_)
            op.launch = [fp, pairs](cudaStream_t st) { trunk_fused_kernel<256, B><<<2 * pairs, kFtThreads, FtG<256, B>::kSmemBytes, st>>>(fp); };
        else if (d_.f == 64)
            op.launch = [fp, pairs](cudaStream_t st) { trunk_fused_kernel<64, E8><<<2 * pairs, kFtThreads, FtG<64, E8>::kSmemBytes, st>>>(fp); };
        else if (d_.f == 128)
            op.launch = [fp, pairs](cudaStream_t st) { trunk_fused_kernel<128, E8><<<2 * pairs, kFtThreads, FtG<128, E8>::kSmemBytes, st>>>(fp); };
        else
            op.launch = [fp, pairs](cudaStream_t st) { trunk_fused_kernel<256, E8><<<2 * pairs, kFtThreads, FtG<256, E8>::kSmemBytes, st>>>(fp); };
        ops.push_back(op);
    } else if (small) {
        // encode + stem + all residual blocks + both 1x1 head convs in one launch (trunk_small.cuh)
        TrunkSmallParams sp;
        std::memset(&sp, 0, sizeof(sp));
        const int W = static_cast<int>(d_.s) + 1, BP = W * W;
        // Tiles per CTA (T) and tiles per independent group: the fewest tiles that still fit the batch on the SMs in
        // one wave (small batches spread out for latency); groups of whole boards, preferring >= 2 groups so that one
        // group's epilogue hides behind another group's MMAs.
        auto plan = [&](int cand, int& tpg, int& per_group) {
            double best = -1.0;
            for (int g = 1; g <= cand; g *= 2) {
                const int bpg = g * 128 / BP, groups = cand / g;
                // single-tile groups keep only 2 accumulator chains in flight (MMA latency-bound): mild penalty
                const double score = static_cast<double>(bpg) * groups * (groups >= 2 ? 1.0 : 0.6) * (g == 1 && cand > 1 ? 0.9 : 1.0);
                if (bpg >= 1 && score > best) {
                    best = score;
                    tpg = g;
                    per_group = bpg;
                }
            }
            return best > 0.0;
        };
        int T = kTsMaxTiles, tpg = kTsMaxTiles, bpg = 0;
        // One tile per CTA gives the lowest latency for a batch that is alone on the GPU, but costs ~2.6x the SM time
        // per position (per-CTA setup, latency-bound MMA chains).  Self-play keeps many batches of 100-300 positions in
        // flight at once (one per worker thread), where that SM time is the bottleneck: measured 16 threads, hex5:
        // 17.4 M sims/s with 1 tile, 18.2 M with >= 2, 17.8 M with >= 4 (no cache: 15.5 M vs 18.0 M with >= 4).
        int min_tiles = bucket >= 128 ? 2 : 1;
        if (const char* e = std::getenv("CATTUS_B200_TRUNK_MIN_TILES")) min_tiles = std::max(1, std::atoi(e));  // experiment knob
        for (int cand = min_tiles; cand <= kTsMaxTiles; cand *= 2) {
            int g = 0, b = 0;
            if (!plan(cand, g, b)) continue;
            const int per_round = b * (cand / g);
            if (cand == kTsMaxTiles || static_cast<int>(ceil_div(bucket, static_cast<uint32_t>(per_round))) <= sm) {
                T = cand;
                tpg = g;
                bpg = b;
                break;
            }
        }
        if (bpg == 0) throw Error(CATTUS_B200_EINVAL, "trunk_small: board does not fit a tile group");
        sp.recs = recs;
        sp.n_ptr = n_ptr;
        sp.wimg = small_w_.as<uint4>();
        sp.bias = small_b_.as<float>();
        sp.out_v = lane.d_hv.as<__nv_bfloat16>();
        sp.out_p = lane.d_hp.as<__nv_bfloat16>();
        sp.err = d_err_;
        if (std::getenv("CATTUS_B200_TRACE_TRUNK")) {  // diagnostic: per-layer clock64 trace of CTA 0, printed by time_stage
            if (trace_.p == nullptr) trace_.alloc(512 * sizeof(unsigned long long));
            sp.dbg = trace_.as<unsigned long long>();
        }
        sp.rec_bytes = rec_.rec_bytes;
        sp.planes = static_cast<int>(d_.c_in);
        sp.wpp = rec_.wpp;
        sp.s = static_cast<int>(d_.s);
        sp.layers = 1 + 2 * static_cast<int>(d_.r);
        sp.stem_kc = static_cast<int>(small_stem_kc_);
        sp.vhp = static_cast<int>(vhp_);
        sp.php = static_cast<int>(php_);
        sp.tiles = T;
        sp.group_tiles = tpg;
        sp.boards_per_group = bpg;
        sp.boards_per_round = bpg * (T / tpg);
        sp.num_rounds = static_cast<int>(ceil_div(bucket, static_cast<uint32_t>(sp.boards_per_round)));
        sp.w_bytes = static_cast<int>((small_stem_kc_ + 2 * d_.r) * 9 * kTsTapBytes + (vhp_ + php_) * 32);
        sp.margin = (W + 1 + 7) / 8 * 8;
        const TsSmemLayout lay = ts_smem_layout(sp.tiles, sp.stem_kc, sp.margin, sp.w_bytes);
        if (lay.total > 200 * 1024) throw Error(CATTUS_B200_EINVAL, "trunk_small: network does not fit in shared memory");
        const int grid = std::min(sm, sp.num_rounds);
        const int smem_bytes = lay.total;
        Op op;
        op.stage = 1;
        op.name = "trunk_small";
        op.launch = [sp, grid, smem_bytes](cudaStream_t st) { trunk_small_kernel<<<grid, kTsThreads, smem_bytes, st>>>(sp); };
        ops.push_back(op);
    } else {
        conv3("stem", x, cin_pad_, convs_[0], nullptr, act[0]);
        for (uint32_t i = 0; i < d_.r; ++i) {
            const int h = (cur + 1) % 3, o = (cur + 2) % 3;
            conv3("block_conv1", act[cur], ca_, convs_[1 + 2 * i], nullptr, act[h]);
            conv3("block_conv2", act[h], ca_, convs_[2 + 2 * i], act[cur], act[o]);
            cur = o;
        }
    }
    if (!small && !fused) {
        gemm(2, "value_conv", act[cur], ca_, rows_total, ca_ * 2ull, vconv_, lane.d_hv.p, vhp_, false, true);
        gemm(2, "policy_conv", act[cur], ca_, rows_total, ca_ * 2ull, pconv_, lane.d_hp.p, php_, false, true);
    }
    // Tails fused into the FC epilogues (flags bit 0 keeps the separate tail kernels as the independent comparison path):
    // value: always (the 128 hidden units are one N tile); policy: when all moves fit one N tile (tic-tac-toe, hex).
    const bool fuse_tails = (desc_.flags & 1u) == 0;
    const bool fuse_policy = fuse_tails && !dense_input && pfc_.n_tiles == 1;
    TcGemmParams value_tc;
    std::memset(&value_tc, 0, sizeof(value_tc));
    gemm(2, "value_fc1", lane.d_hv.p, static_cast<uint64_t>(s2) * vhp_, bucket, static_cast<uint64_t>(s2) * vhp_ * 2, vfc1_, lane.d_hidden.p, 128,
         true, true);
    if (fuse_tails) {
        Op& op = ops.back();
        TcGemmParams p = last_tc;
        p.epi = 1;
        p.w2 = vfc2_w_.as<float>();
        p.b2 = vfc2_b_;
        p.values = zero_copy_out(lane, bucket, dense_input) ? lane.zc_values : lane.d_values.as<float>();
        p.n_ptr = n_ptr;
        op = make_tc_op(2, "value_fc1_tanh", p, ceil_div(bucket, 128), 1);
        value_tc = p;
    }
    gemm(2, "policy_fc", lane.d_hp.p, static_cast<uint64_t>(s2) * php_, bucket, static_cast<uint64_t>(s2) * php_ * 2, pfc_, lane.d_logits.p,
         pfc_.n_umma * pfc_.n_tiles, true, false);
    const bool compact_policy = fuse_tails && !dense_input && pfc_.n_tiles > 1 && pfc_.n_umma == 128 && d_.moves <= 256 * 32;
    if (fuse_policy || compact_policy) {
        Op& op = ops.back();
        TcGemmParams p = last_tc;
        p.epi = fuse_policy ? 2 : 3;
        p.recs = recs;
        p.rl = L;
        p.probs = zero_copy_out(lane, bucket, dense_input) ? lane.zc_probs : lane.d_probs.as<float>();
        p.n_ptr = n_ptr;
        op = make_tc_op(2, fuse_policy ? "policy_fc_softmax" : "policy_fc_masked", p, ceil_div(bucket, 128), pfc_.n_tiles);
    }
    if (fuse_tails && (fuse_policy || compact_policy)) {
        // both FCs in one launch (tc_gemm_dual_kernel): y == 0 value, y >= 1 the policy's N tiles
        TcGemmDualParams dp;
        dp.b = last_tc;  // still the policy problem ...
        dp.b.epi = fuse_policy ? 2 : 3;
        dp.b.recs = recs;
        dp.b.rl = L;
        // the masked logits of epi 3 stay in HBM: softmax_compact reads them there and writes the probabilities to wherever
        // the caller reads them (zero-copy host memory for small buckets -- no read has to cross PCIe)
        dp.b.probs = compact_policy || !zero_copy_out(lane, bucket, dense_input) ? lane.d_probs.as<float>() : lane.zc_probs;
        dp.b.n_ptr = n_ptr;
        dp.a = value_tc;
        ops.pop_back();
        ops.pop_back();
        Op op;
        op.stage = 2;
        op.name = "heads_fc_dual";
        const dim3 grid(ceil_div(bucket, 128), 1 + pfc_.n_tiles);
        // the deep form needs an even number of k-blocks in BOTH problems (an odd one falls back to the 3-stage ring)
        const int kb_both = (dp.a.num_kb % 2 == 0 && dp.b.num_kb % 2 == 0) ? std::max(dp.a.num_kb, dp.b.num_kb) : 1;
        const int stages = tc_stages_for(grid.x * grid.y, kb_both, bucket);
        dp.a.fault = (desc_.flags & 2u) ? 1 : 0;
        if (std::getenv("CATTUS_B200_TRACE_HEADS")) {  // diagnostic: clock64 trace of the policy FC's tile (0, 1), printed by time_stage
            if (trace_.p == nullptr) trace_.alloc(512 * sizeof(unsigned long long));
            dp.a.dbg = dp.b.dbg = trace_.as<unsigned long long>();
        }
        const int smem_bytes = tc_smem_bytes(stages);
        if (stages == kTcStagesDeep)
            op.launch = [dp, grid, smem_bytes](cudaStream_t st) { launch_pdl(tc_gemm_dual_kernel<2>, grid, dim3(kTcThreads), smem_bytes, st, dp); };
        else
            op.launch = [dp, grid, smem_bytes](cudaStream_t st) { launch_pdl(tc_gemm_dual_kernel<1>, grid, dim3(kTcThreads), smem_bytes, st, dp); };
        ops.push_back(op);
    }
    if (compact_policy) {
        Op op;
        op.stage = 3;
        op.name = "softmax_compact";
        const float* logits = lane.d_probs.as<float>();
        float* probs = zero_copy_out(lane, bucket, dense_input) ? lane.zc_probs : lane.d_probs.as<float>();
        const int blocks = static_cast<int>(ceil_div(bucket * 32, 256));
        op.launch = [=](cudaStream_t st) { launch_pdl(softmax_compact_kernel, dim3(blocks), dim3(256), 0, st, recs, L, n_ptr, logits, probs); };
        ops.push_back(op);
    }
    add_tail_ops(lane, bucket, ops, dense_input, !fuse_tails, !(fuse_policy || compact_policy));
}

void Engine::run_bucket(Lane& lane, uint32_t bucket, cudaStream_t stream, bool use_graph, bool dense_input) {
    std::vector<Op>& ops = ops_for(lane, bucket, dense_input);
    if (!use_graph) {
        for (const Op& op : ops) op.launch(stream);
        CB2_CUDA(cudaGetLastError());
        return;
    }
    const uint32_t key = bucket | (dense_input ? 0x80000000u : 0u) | (lane.device_out ? 0x40000000u : 0u);
    auto it = lane.graphs.find(key);
    if (it == lane.graphs.end()) {
        // capture on the lane's own stream (never on a caller's stream)
        cudaGraph_t graph = nullptr;
        CB2_CUDA(cudaStreamBeginCapture(lane.stream, cudaStreamCaptureModeThreadLocal));
        try {
            for (const Op& op : ops) op.launch(lane.stream);
        } catch (...) {  // a launch that throws (launch_pdl checks its result) must not leave the stream capturing
            cudaStreamEndCapture(lane.stream, &graph);
            if (graph) cudaGraphDestroy(graph);
            throw;
        }
        cudaError_t ce = cudaStreamEndCapture(lane.stream, &graph);
        if (ce != cudaSuccess) throw Error(CATTUS_B200_ECUDA, std::string("graph capture failed: ") + cudaGetErrorString(ce));
        cudaGraphExec_t exec = nullptr;
        ce = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ce != cudaSuccess) throw Error(CATTUS_B200_ECUDA, std::string("graph instantiate failed: ") + cudaGetErrorString(ce));
        it = lane.graphs.emplace(key, exec).first;
    }
    CB2_CUDA(cudaGraphLaunch(it->second, stream));
}

void Engine::throw_device_error(const char* where, cudaError_t e) {
    const uint32_t code = h_err_ ? *h_err_ : 0;
    char buf[256];
    std::snprintf(buf, sizeof(buf), "%s: %s (device fault word 0x%x)", where, cudaGetErrorString(e), code);
    throw Error(code ? CATTUS_B200_EDEVICE : CATTUS_B200_ECUDA, buf);
}

// ------------------------------------------------------------------------------------------------ pack pool
PackPool::PackPool(unsigned helpers) {
    for (unsigned i = 0; i < helpers; ++i) threads_.emplace_back([this] { worker(); });
}
PackPool::~PackPool() {
    {
        std::lock_guard<std::mutex> g(mu_);
        stop_ = true;
    }
    cv_.notify_all();
    for (auto& t : threads_) t.join();
}
void PackPool::worker() {
    uint64_t seen = 0;
    for (;;) {
        const std::function<void(int)>* job;
        int slices;
        {
            std::unique_lock<std::mutex> g(mu_);
            cv_.wait(g, [&] { return stop_ || gen_ != seen; });
            if (stop_) return;
            seen = gen_;
            if (job_ == nullptr) continue;  // woke up after that run was over
            job = job_;
            slices = slices_;
            ++active_;  // try_run does not return (and the next run cannot reset next_) while a helper holds its job
        }
        int done = 0;
        for (int i; (i = next_.fetch_add(1)) < slices;) {
            (*job)(i);
            ++done;
        }
        {
            std::lock_guard<std::mutex> g(mu_);
            remaining_ -= done;
            --active_;
            if (remaining_ == 0 && active_ == 0) done_cv_.notify_all();
        }
    }
}
bool PackPool::try_run(int slices, const std::function<void(int)>& fn) {
    std::unique_lock<std::mutex> run(run_mu_, std::try_to_lock);
    if (!run.owns_lock()) return false;
    {
        std::lock_guard<std::mutex> g(mu_);
        job_ = &fn;
        slices_ = slices;
        remaining_ = slices;
        next_.store(0);
        ++gen_;
    }
    cv_.notify_all();
    int done = 0;
    for (int i; (i = next_.fetch_add(1)) < slices;) {
        fn(i);
        ++done;
    }
    std::unique_lock<std::mutex> g(mu_);
    remaining_ -= done;
    done_cv_.wait(g, [&] { return remaining_ == 0 && active_ == 0; });
    job_ = nullptr;
    return true;
}

// ------------------------------------------------------------------------------------------------ batches
uint32_t Engine::pack_record(uint8_t* dst, const uint64_t* planes, const uint8_t* legal, uint32_t prob_offset) const {
    const int plane_bytes = rec_.planes * rec_.wpp * 8;
    std::memcpy(dst, planes, plane_bytes);
    uint32_t cnt = 0;
    if (derive_legal_) {
        for (int k = 0; k < rec_.wpp; ++k) {
            uint64_t e = planes[2 * rec_.wpp + k] & ~(planes[k] | planes[rec_.wpp + k]);
            const int rem = rec_.moves - 64 * k;
            if (rem < 64) e &= (rem <= 0) ? 0ull : ((1ull << rem) - 1ull);
            cnt += static_cast<uint32_t>(__builtin_popcountll(e));
        }
    } else {
        if (legal == nullptr) throw Error(CATTUS_B200_EINVAL, "this game needs an explicit legal-move bitmap");
        const int bm = static_cast<int>(d_.bitmap_bytes());
        const int padded = rec_.rec_bytes - kRecPrefix - plane_bytes;
        uint8_t* d = dst + plane_bytes;
        std::memcpy(d, legal, bm);
        std::memset(d + bm, 0, padded - bm);
        if (rec_.moves % 8) d[bm - 1] &= static_cast<uint8_t>((1u << (rec_.moves % 8)) - 1u);
        const uint64_t* w = reinterpret_cast<const uint64_t*>(d);
        for (int k = 0; k < padded / 8; ++k) cnt += static_cast<uint32_t>(__builtin_popcountll(w[k]));
        // softmax_compact_kernel holds at most 8 x 32 logits per position; the reference's serializer caps a chess position at
        // 225 legal moves (serialize/chess.rs:34) and no legal position exceeds 218
        if (cnt > 256) throw Error(CATTUS_B200_ERANGE, "legal bitmap with " + std::to_string(cnt) + " moves set (at most 256 per position)");
    }
    uint32_t* prefix = reinterpret_cast<uint32_t*>(dst - kRecPrefix);
    prefix[0] = prob_offset;
    prefix[1] = cnt;
    return cnt;
}

void Engine::submit(Lane& l, uint32_t n, uint32_t total_probs) {
    *reinterpret_cast<uint32_t*>(l.h_in) = n;
    CB2_CUDA(cudaMemcpyAsync(l.d_in.p, l.h_in, 16 + static_cast<size_t>(n) * rec_.rec_bytes, cudaMemcpyHostToDevice, l.stream));
    run_bucket(l, bucket_for(n), l.stream, true, false);
    if (!zero_copy_out(l, bucket_for(n), false)) {  // small batches wrote h_values / h_probs directly (mapped pinned memory)
        CB2_CUDA(cudaMemcpyAsync(l.h_values, l.d_values.p, sizeof(float) * n, cudaMemcpyDeviceToHost, l.stream));
        if (total_probs) CB2_CUDA(cudaMemcpyAsync(l.h_probs, l.d_probs.p, sizeof(float) * total_probs, cudaMemcpyDeviceToHost, l.stream));
    }
    CB2_CUDA(cudaEventRecord(l.done, l.stream));
}

void Engine::finish(Lane& l, uint32_t n) {
    cudaError_t e = cudaEventSynchronize(l.done);
    if (e != cudaSuccess) throw_device_error("batch", e);
    (void)n;
}

Lane& Engine::acquire_lane() {
    std::unique_lock<std::mutex> g(lane_mu_);
    for (;;) {
        for (size_t i = 0; i < lanes_.size(); ++i)
            if (!lane_busy_[i]) {
                lane_busy_[i] = 1;
                return *lanes_[i];
            }
        lane_cv_.wait(g);
    }
}
Lane* Engine::try_acquire_lane() {
    std::lock_guard<std::mutex> g(lane_mu_);
    for (size_t i = 0; i < lanes_.size(); ++i)
        if (!lane_busy_[i]) {
            lane_busy_[i] = 1;
            return lanes_[i].get();
        }
    return nullptr;
}
void Engine::release_lane(Lane& l) {
    {
        std::lock_guard<std::mutex> g(lane_mu_);
        lane_busy_[l.index] = 0;
    }
    lane_cv_.notify_one();
}

void Engine::note_batch(uint32_t n, double seconds) {
    std::lock_guard<std::mutex> g(m_mu_);
    metrics_.activation_count += 1;
    metrics_.positions += n;
    metrics_.run_duration_last = seconds;
    // RunningAverage(0.99): engine/src/util/metric.rs:1-20 -- value starts at 0, then value = (1 - e) * value + e * x
    metrics_.run_duration_ema = metrics_.run_duration_ema * (1.0 - 0.99) + seconds * 0.99;
    metrics_.mean_batch_fill = static_cast<double>(metrics_.positions) / (static_cast<double>(metrics_.activation_count) * max_batch_);
    metrics_.kernel_launches += kernels_per_batch_;
}

// The per-leaf path.  A worker writes its record into the open pinned block under the queue lock, then sleeps on a
// condition variable until an evaluator thread has shipped the block and scattered the results back.
void Engine::eval_leaf(const uint64_t* planes, const uint8_t* legal, LeafRequest* req) {
    std::unique_lock<std::mutex> g(q_mu_);
    q_space_cv_.wait(g, [&] { return stopping_ || open_reqs_.size() < max_batch_; });
    if (stopping_) throw Error(CATTUS_B200_EINVAL, "evaluator is shutting down");
    const uint32_t slot = static_cast<uint32_t>(open_reqs_.size());
    req->count = pack_record(open_block_ + kRecs0 + static_cast<size_t>(slot) * rec_.rec_bytes, planes, legal, open_total_);
    if (req->count > req->probs_cap) throw Error(CATTUS_B200_ERANGE, "probs_cap is smaller than the number of legal moves");
    req->status = 1;
    open_reqs_.push_back(req);
    open_total_ += req->count;
    open_count_.store(static_cast<uint32_t>(open_reqs_.size()), std::memory_order_release);
    g.unlock();
    q_cv_.notify_one();
    // A condition-variable wake-up costs 10-30 us, a third of a whole small-batch round trip: spin on the request's
    // flag for about as long as a batch takes, then fall back to sleeping.
    const auto spin_until = std::chrono::steady_clock::now() + std::chrono::microseconds(400);
    for (uint32_t i = 0; req->done.load(std::memory_order_acquire) == 0; ++i) {
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
        if ((i & 63u) == 63u && std::chrono::steady_clock::now() > spin_until) {
            g.lock();
            done_cv_.wait(g, [&] { return req->status != 1; });
            g.unlock();
            break;
        }
    }
    if (req->status < 0) throw Error(req->status, req->error);
}

void Engine::evaluator_loop() {
    cudaSetDevice(device_);
    std::vector<LeafRequest*> reqs;
    for (;;) {
        {
            // stay hot for a moment after the last batch (per-leaf callers come back within microseconds), then sleep
            const auto spin_until = std::chrono::steady_clock::now() + std::chrono::microseconds(200);
            for (uint32_t i = 0; open_count_.load(std::memory_order_acquire) == 0; ++i) {
#if defined(__x86_64__)
                __builtin_ia32_pause();
#endif
                if ((i & 63u) == 63u && std::chrono::steady_clock::now() > spin_until) break;
            }
            std::unique_lock<std::mutex> g(q_mu_);
            q_cv_.wait(g, [&] { return stopping_ || !open_reqs_.empty(); });
            if (stopping_ && open_reqs_.empty()) return;
        }
        Lane& l = acquire_lane();
        uint32_t total = 0;
        {
            std::lock_guard<std::mutex> g(q_mu_);
            if (open_reqs_.empty()) {  // another evaluator took the block while we waited for a lane
                release_lane(l);
                continue;
            }
            std::swap(open_block_, l.h_in);
            reqs.swap(open_reqs_);
            open_reqs_.clear();
            open_count_.store(0, std::memory_order_release);
            total = open_total_;
            open_total_ = 0;
        }
        q_space_cv_.notify_all();
        const uint32_t n = static_cast<uint32_t>(reqs.size());
        int status = 0;
        std::string err;
        const auto t0 = std::chrono::steady_clock::now();
        try {
            submit(l, n, total);
            finish(l, n);
            note_batch(n, std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
        } catch (const Error& e) {
            status = e.code;
            err = e.what();
        }
        {
            std::lock_guard<std::mutex> g(q_mu_);
            uint32_t off = 0;
            for (uint32_t i = 0; i < n; ++i) {
                LeafRequest* r = reqs[i];
                if (status == 0) {
                    std::memcpy(r->probs_out, l.h_probs + off, sizeof(float) * r->count);
                    *r->n_probs = r->count;
                    *r->value_out = l.h_values[i];
                    r->status = 0;
                } else {
                    r->error = err;
                    r->status = status;
                }
                off += r->count;
                r->done.store(1, std::memory_order_release);  // r may be gone the moment a spinning caller sees this
            }
        }
        done_cv_.notify_all();
        reqs.clear();
        release_lane(l);
    }
}

// Synchronous bulk path: chunks of max_batch pipelined over the lanes (pack chunk i+1 while chunk i runs).
void Engine::eval_batch(const uint64_t* planes, const uint8_t* legal, uint32_t n, float* probs_out, size_t probs_cap, uint32_t* prob_offsets,
                        float* values_out) {
    if (n == 0) {
        if (prob_offsets) prob_offsets[0] = 0;
        return;
    }
    if (!planes || !probs_out || !prob_offsets || !values_out) throw Error(CATTUS_B200_EINVAL, "null argument");
    CB2_CUDA(cudaSetDevice(device_));
    struct InFlight {
        Lane* lane;
        uint32_t first, n, total;
        size_t prob_base;
        std::chrono::steady_clock::time_point t0;
    };
    std::deque<InFlight> inflight;
    static const bool trace = std::getenv("CATTUS_B200_TRACE_BATCH") != nullptr;  // diagnostic timeline on stderr
    const auto call_t0 = std::chrono::steady_clock::now();
    auto stamp = [&](const char* what, uint32_t first) {
        if (trace) std::fprintf(stderr, "eval_batch %8.1f us  %s %u\n", std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - call_t0).count(), what, first);
    };
    const size_t plane_words = static_cast<size_t>(rec_.planes) * rec_.wpp;
    const size_t bm = d_.bitmap_bytes();
    size_t prob_cursor = 0;
    auto drain_one = [&]() {
        InFlight f = inflight.front();
        inflight.pop_front();
        try {
            stamp("drain wait", f.first);
            finish(*f.lane, f.n);
            stamp("drain done", f.first);
        } catch (...) {
            release_lane(*f.lane);  // the other chunks may still be executing: the caller's handler waits for them first
            throw;
        }
        std::memcpy(values_out + f.first, f.lane->h_values, sizeof(float) * f.n);
        std::memcpy(probs_out + f.prob_base, f.lane->h_probs, sizeof(float) * f.total);
        note_batch(f.n, std::chrono::duration<double>(std::chrono::steady_clock::now() - f.t0).count());
        release_lane(*f.lane);
        stamp("copied out", f.first);
    };
    try {
        // A call of several device batches ramps in and out with a quarter-size chunk: the GPU starts after a quarter of
        // the first batch is packed and copied, and the last results to copy back are a quarter batch -- the pipeline's fill
        // and drain are what an end-to-end call loses against resident inputs.
        const uint32_t quarter = std::max<uint32_t>(64, max_batch_ / 4);
        const bool ramp = n > max_batch_ && lanes_.size() >= 2 && max_batch_ >= 256;
        uint32_t cn = 0;
        for (uint32_t first = 0; first < n; first += cn) {
            const uint32_t left = n - first;
            cn = std::min(max_batch_, left);
            if (ramp) {
                if (first == 0)
                    cn = quarter;
                else if (left > quarter && left <= max_batch_ + quarter)
                    cn = left - quarter;  // leaves exactly one quarter chunk for the end
            }
            if (inflight.size() >= lanes_.size()) drain_one();
            Lane& l = acquire_lane();
            uint32_t total = 0;
            try {
                auto pack_range = [&](uint32_t lo, uint32_t hi) {  // offsets relative to `lo`'s first probability
                    uint32_t run = 0;
                    for (uint32_t i = lo; i < hi; ++i) {
                        const uint32_t b = first + i;
                        const uint32_t c = pack_record(l.h_in + kRecs0 + static_cast<size_t>(i) * rec_.rec_bytes, planes + b * plane_words,
                                                       legal ? legal + b * bm : nullptr, run);
                        prob_offsets[b] = run;
                        run += c;
                    }
                    return run;
                };
                constexpr uint32_t kSlices = 8;
                uint32_t slice_total[kSlices] = {0};
                std::string slice_error;
                int slice_code = 0;
                const uint32_t per = (cn + kSlices - 1) / kSlices;
                const std::function<void(int)> job = [&](int sl) {
                    const uint32_t lo = std::min(cn, static_cast<uint32_t>(sl) * per), hi = std::min(cn, lo + per);
                    try {
                        slice_total[sl] = pack_range(lo, hi);
                    } catch (const Error& e) {
                        std::lock_guard<std::mutex> g(m_mu_);
                        slice_code = e.code;
                        slice_error = e.what();
                    }
                };
                if (cn >= 1024 && pack_pool_ && pack_pool_->try_run(static_cast<int>(kSlices), job)) {
                    if (slice_code) throw Error(slice_code, slice_error);
                    uint32_t base = 0;  // turn slice-relative offsets into chunk-relative (record prefix) and call-relative (output)
                    for (uint32_t sl = 0; sl < kSlices; ++sl) {
                        const uint32_t lo = std::min(cn, sl * per), hi = std::min(cn, lo + per);
                        for (uint32_t i = lo; i < hi; ++i) {
                            *reinterpret_cast<uint32_t*>(l.h_in + kRecs0 + static_cast<size_t>(i) * rec_.rec_bytes - kRecPrefix) += base;
                            prob_offsets[first + i] += static_cast<uint32_t>(prob_cursor) + base;
                        }
                        base += slice_total[sl];
                    }
                    total = base;
                } else {
                    total = pack_range(0, cn);
                    for (uint32_t i = 0; i < cn; ++i) prob_offsets[first + i] += static_cast<uint32_t>(prob_cursor);
                }
                if (prob_cursor + total > probs_cap) throw Error(CATTUS_B200_ERANGE, "probs_cap is smaller than the number of legal moves");
                InFlight f{&l, first, cn, total, prob_cursor, std::chrono::steady_clock::now()};
                stamp("packed", first);
                submit(l, cn, total);
                stamp("submitted", first);
                inflight.push_back(f);
            } catch (...) {
                release_lane(l);
                throw;
            }
            prob_cursor += total;
        }
        prob_offsets[n] = static_cast<uint32_t>(prob_cursor);
        while (!inflight.empty()) drain_one();
    } catch (...) {
        while (!inflight.empty()) {
            cudaEventSynchronize(inflight.front().lane->done);
            release_lane(*inflight.front().lane);
            inflight.pop_front();
        }
        throw;
    }
}

// Split form of eval_batch for one device batch: lets a caller keep several batches in flight (the self-play driver
// simulates one group of games while another group's leaves are on the GPU).
int Engine::eval_batch_submit(const uint64_t* planes, const uint8_t* legal, uint32_t n, bool block) {
    if (n == 0 || n > max_batch_) throw Error(CATTUS_B200_ERANGE, "eval_batch_submit: n must be 1..max_batch");
    if (!planes) throw Error(CATTUS_B200_EINVAL, "null argument");
    CB2_CUDA(cudaSetDevice(device_));
    Lane* lp = block ? &acquire_lane() : try_acquire_lane();
    if (lp == nullptr) return -1;
    Lane& l = *lp;
    try {
        const size_t plane_words = static_cast<size_t>(rec_.planes) * rec_.wpp;
        const size_t bm = d_.bitmap_bytes();
        l.async_counts.resize(n);
        uint32_t total = 0;
        for (uint32_t i = 0; i < n; ++i) {
            const uint32_t c = pack_record(l.h_in + kRecs0 + static_cast<size_t>(i) * rec_.rec_bytes, planes + i * plane_words, legal ? legal + i * bm : nullptr, total);
            l.async_counts[i] = c;
            total += c;
        }
        l.async_n = n;
        l.async_total = total;
        l.async_t0 = std::chrono::steady_clock::now();
        submit(l, n, total);
    } catch (...) {
        release_lane(l);
        throw;
    }
    return l.index;
}

void Engine::eval_batch_wait(int ticket, float* probs_out, size_t probs_cap, uint32_t* prob_offsets, float* values_out) {
    if (ticket < 0 || ticket >= static_cast<int>(lanes_.size())) throw Error(CATTUS_B200_EINVAL, "eval_batch_wait: bad ticket");
    Lane& l = *lanes_[ticket];
    if (l.async_n == 0) throw Error(CATTUS_B200_EINVAL, "eval_batch_wait: nothing in flight on this ticket");
    const uint32_t n = l.async_n, total = l.async_total;
    try {
        if (!probs_out || !prob_offsets || !values_out) throw Error(CATTUS_B200_EINVAL, "null argument");
        if (total > probs_cap) throw Error(CATTUS_B200_ERANGE, "probs_cap is smaller than the number of legal moves");
        finish(l, n);
        uint32_t run = 0;
        for (uint32_t i = 0; i < n; ++i) {
            prob_offsets[i] = run;
            run += l.async_counts[i];
        }
        prob_offsets[n] = run;
        std::memcpy(values_out, l.h_values, sizeof(float) * n);
        std::memcpy(probs_out, l.h_probs, sizeof(float) * total);
        note_batch(n, std::chrono::duration<double>(std::chrono::steady_clock::now() - l.async_t0).count());
    } catch (...) {
        cudaEventSynchronize(l.done);
        l.async_n = 0;
        release_lane(l);
        throw;
    }
    l.async_n = 0;
    release_lane(l);
}

void Engine::encode(const uint64_t* planes, uint32_t n, uint32_t batch, float* nchw_out) {
    if (n < 1 || n > batch) throw Error(CATTUS_B200_EINVAL, "invalid sample len " + std::to_string(n) + ", 1..=" + std::to_string(batch));
    if (batch > max_batch_) throw Error(CATTUS_B200_ERANGE, "batch_size exceeds max_batch");
    CB2_CUDA(cudaSetDevice(device_));
    Lane& l = acquire_lane();
    try {
        const size_t plane_bytes = static_cast<size_t>(rec_.planes) * rec_.wpp * 8;
        for (uint32_t i = 0; i < n; ++i) {
            uint8_t* dst = l.h_in + kRecs0 + static_cast<size_t>(i) * rec_.rec_bytes;
            std::memset(dst - kRecPrefix, 0, rec_.rec_bytes);
            std::memcpy(dst, planes + i * (plane_bytes / 8), plane_bytes);
        }
        *reinterpret_cast<uint32_t*>(l.h_in) = n;
        CB2_CUDA(cudaMemcpyAsync(l.d_in.p, l.h_in, 16 + static_cast<size_t>(n) * rec_.rec_bytes, cudaMemcpyHostToDevice, l.stream));
        const long long total = static_cast<long long>(batch) * d_.c_in * d_.s2();
        encode_nchw_f32_kernel<<<grid_for(total, 256, sm_count_), 256, 0, l.stream>>>(l.d_in.as<uint8_t>() + kRecs0, rec_, l.d_in.as<uint32_t>(),
                                                                                     static_cast<int>(batch), l.d_dense.as<float>());
        CB2_CUDA(cudaGetLastError());
        CB2_CUDA(cudaMemcpyAsync(nchw_out, l.d_dense.p, sizeof(float) * total, cudaMemcpyDeviceToHost, l.stream));
        cudaError_t e = cudaStreamSynchronize(l.stream);
        if (e != cudaSuccess) throw_device_error("encode", e);
        {
            std::lock_guard<std::mutex> g(m_mu_);
            metrics_.kernel_launches += 1;
        }
    } catch (...) {
        release_lane(l);
        throw;
    }
    release_lane(l);
}

void Engine::run_dense(const float* nchw, uint32_t n, float* logits_out, float* values_out) {
    if (fp8_) throw Error(CATTUS_B200_EINVAL, "run_dense: there is no dense-input path at precision FP8 (the FP8 trunk reads packed bitboards); "
                                              "use a BF16 or FP32_CHECK handle");
    if (n == 0) return;
    if (!nchw || !logits_out || !values_out) throw Error(CATTUS_B200_EINVAL, "null argument");
    CB2_CUDA(cudaSetDevice(device_));
    const size_t per = static_cast<size_t>(d_.c_in) * d_.s2();
    const uint32_t ld = precision_ == CATTUS_B200_PRECISION_FP32_CHECK ? d_.moves : pfc_.n_umma * pfc_.n_tiles;
    Lane& l = acquire_lane();
    try {
        for (uint32_t first = 0; first < n; first += max_batch_) {
            const uint32_t cn = std::min(max_batch_, n - first);
            const uint32_t bucket = bucket_for(cn);
            *reinterpret_cast<uint32_t*>(l.h_in) = cn;
            CB2_CUDA(cudaMemcpyAsync(l.d_in.p, l.h_in, 16, cudaMemcpyHostToDevice, l.stream));
            if (bucket > cn) CB2_CUDA(cudaMemsetAsync(l.d_dense.as<float>() + cn * per, 0, sizeof(float) * (bucket - cn) * per, l.stream));
            CB2_CUDA(cudaMemcpyAsync(l.d_dense.p, nchw + first * per, sizeof(float) * cn * per, cudaMemcpyHostToDevice, l.stream));
            run_bucket(l, bucket, l.stream, true, true);
            CB2_CUDA(cudaMemcpy2DAsync(logits_out + static_cast<size_t>(first) * d_.moves, sizeof(float) * d_.moves, l.d_logits.p, sizeof(float) * ld,
                                       sizeof(float) * d_.moves, cn, cudaMemcpyDeviceToHost, l.stream));
            CB2_CUDA(cudaMemcpyAsync(values_out + first, l.d_values.p, sizeof(float) * cn, cudaMemcpyDeviceToHost, l.stream));
            cudaError_t e = cudaStreamSynchronize(l.stream);
            if (e != cudaSuccess) throw_device_error("run_dense", e);
            std::lock_guard<std::mutex> g(m_mu_);
            metrics_.kernel_launches += ops_for(l, bucket, true).size();
        }
    } catch (...) {
        release_lane(l);
        throw;
    }
    release_lane(l);
}

// Device-resident variant (lane 0): used by the bench to time the kernels with inputs already in HBM.
void Engine::resident_upload(const uint64_t* planes, const uint8_t* legal, uint32_t n) {
    if (n == 0 || n > max_batch_) throw Error(CATTUS_B200_ERANGE, "resident batch must be 1..max_batch");
    CB2_CUDA(cudaSetDevice(device_));
    Lane& l = *lanes_[0];
    const size_t plane_words = static_cast<size_t>(rec_.planes) * rec_.wpp;
    const size_t bm = d_.bitmap_bytes();
    resident_offsets_.assign(n + 1, 0);
    uint32_t total = 0;
    for (uint32_t i = 0; i < n; ++i) {
        resident_offsets_[i] = total;
        total += pack_record(l.h_in + kRecs0 + static_cast<size_t>(i) * rec_.rec_bytes, planes + i * plane_words, legal ? legal + i * bm : nullptr, total);
    }
    resident_offsets_[n] = total;
    *reinterpret_cast<uint32_t*>(l.h_in) = n;
    CB2_CUDA(cudaMemcpyAsync(l.d_in.p, l.h_in, 16 + static_cast<size_t>(n) * rec_.rec_bytes, cudaMemcpyHostToDevice, l.stream));
    CB2_CUDA(cudaStreamSynchronize(l.stream));
}

void Engine::eval_resident(uint32_t n, cudaStream_t stream) {
    if (n == 0 || n > max_batch_) throw Error(CATTUS_B200_ERANGE, "resident batch must be 1..max_batch");
    CB2_CUDA(cudaSetDevice(device_));
    Lane& l = *lanes_[0];
    run_bucket(l, bucket_for(n), stream ? stream : l.stream, true, false);
    std::lock_guard<std::mutex> g(m_mu_);
    metrics_.kernel_launches += kernels_per_batch_;
}

void Engine::resident_download(uint32_t n, float* probs_out, size_t probs_cap, uint32_t* prob_offsets, float* values_out) {
    if (n == 0 || n > max_batch_) throw Error(CATTUS_B200_ERANGE, "resident batch must be 1..max_batch");
    CB2_CUDA(cudaSetDevice(device_));
    Lane& l = *lanes_[0];
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) throw_device_error("eval_resident", e);
    if (resident_offsets_.size() != static_cast<size_t>(n) + 1) throw Error(CATTUS_B200_EINVAL, "resident_download: n differs from the uploaded batch");
    std::memcpy(prob_offsets, resident_offsets_.data(), sizeof(uint32_t) * (n + 1));
    const uint32_t total = prob_offsets[n];
    if (total > probs_cap) throw Error(CATTUS_B200_ERANGE, "probs_cap is smaller than the number of legal moves");
    if (zero_copy_out(l, bucket_for(n), false)) {
        std::memcpy(probs_out, l.h_probs, sizeof(float) * total);
        std::memcpy(values_out, l.h_values, sizeof(float) * n);
    } else {
        CB2_CUDA(cudaMemcpy(probs_out, l.d_probs.p, sizeof(float) * total, cudaMemcpyDeviceToHost));
        CB2_CUDA(cudaMemcpy(values_out, l.d_values.p, sizeof(float) * n, cudaMemcpyDeviceToHost));
    }
}

Engine::ResidentIo Engine::resident_acquire(bool block) {
    CB2_CUDA(cudaSetDevice(device_));
    ResidentIo io;
    Lane* lp = block ? &acquire_lane() : try_acquire_lane();
    if (lp == nullptr) return io;  // lane == -1: every stream is taken
    Lane& l = *lp;
    l.device_out = true;
    io.lane = l.index;
    io.d_block = l.d_in.as<uint8_t>();
    io.d_values = l.d_values.as<float>();
    io.d_probs = l.d_probs.as<float>();
    io.rec_bytes = static_cast<uint32_t>(rec_.rec_bytes);
    io.plane_words = static_cast<uint32_t>(rec_.planes * rec_.wpp);
    io.max_batch = max_batch_;
    io.moves = d_.moves;
    try {
        io.kernels = static_cast<uint32_t>(ops_for(l, bucket_for(max_batch_), false).size());
    } catch (...) {
        l.device_out = false;
        release_lane(l);
        throw;
    }
    return io;
}

void Engine::resident_enqueue(int lane, cudaStream_t stream) {
    Lane& l = *lanes_.at(static_cast<size_t>(lane));
    run_bucket(l, bucket_for(max_batch_), stream, false, false);
}

void Engine::resident_release(int lane) {
    Lane& l = *lanes_.at(static_cast<size_t>(lane));
    l.device_out = false;
    release_lane(l);
}

void Engine::note_resident(uint64_t batches, uint64_t positions, uint64_t launches, double last_seconds) {
    std::lock_guard<std::mutex> g(m_mu_);
    metrics_.activation_count += batches;
    metrics_.positions += positions;
    metrics_.kernel_launches += launches;
    if (batches) {
        metrics_.run_duration_last = last_seconds;
        metrics_.run_duration_ema = metrics_.run_duration_ema * (1.0 - 0.99) + last_seconds * 0.99;
        metrics_.mean_batch_fill = static_cast<double>(metrics_.positions) / (static_cast<double>(metrics_.activation_count) * max_batch_);
    }
}

// ms_out[i] = device time of iteration i of the selected stage(s) on lane 0's stream, CUDA events on that stream,
// with an L2 flush (256 MiB memset) before every iteration, outside the timed bracket.
void Engine::time_stage(uint32_t stage, uint32_t n, uint32_t iters, float* ms_out) {
    if (stage == 5) {
        time_stages_split(n, iters, ms_out);
        return;
    }
    if (n == 0 || n > max_batch_ || iters == 0 || stage > 4) throw Error(CATTUS_B200_EINVAL, "time_stage: bad argument");
    CB2_CUDA(cudaSetDevice(device_));
    Lane& l = *lanes_[0];
    if (flush_.p == nullptr) flush_.alloc(256ull << 20);
    const uint32_t bucket = bucket_for(n);
    std::vector<Op>& ops = ops_for(l, bucket, false);
    std::vector<cudaEvent_t> ev(2 * iters);
    for (auto& e : ev) CB2_CUDA(cudaEventCreate(&e));
    uint64_t launched = 0;
    static const bool no_flush = std::getenv("CATTUS_B200_TIME_NO_FLUSH") != nullptr;  // experiment: weights stay in L2 between iterations
    for (uint32_t it = 0; it < iters; ++it) {
        if (!no_flush) CB2_CUDA(cudaMemsetAsync(flush_.p, static_cast<int>(it & 0xFF), flush_.bytes, l.stream));
        CB2_CUDA(cudaEventRecord(ev[2 * it], l.stream));
        if (stage == 4) {
            static const bool no_graph = std::getenv("CATTUS_B200_TIME_NO_GRAPH") != nullptr;  // experiment: direct launches instead of the graph
            run_bucket(l, bucket, l.stream, !no_graph, false);
            launched += ops.size();
        } else {
            for (const Op& op : ops)
                if (op.stage == static_cast<int>(stage)) {
                    op.launch(l.stream);
                    ++launched;
                }
        }
        CB2_CUDA(cudaEventRecord(ev[2 * it + 1], l.stream));
    }
    cudaError_t e = cudaStreamSynchronize(l.stream);
    if (e != cudaSuccess) throw_device_error("time_stage", e);
    for (uint32_t it = 0; it < iters; ++it) CB2_CUDA(cudaEventElapsedTime(&ms_out[it], ev[2 * it], ev[2 * it + 1]));
    if (trace_.p != nullptr && stage == 1 && std::getenv("CATTUS_B200_TRACE_TRUNK")) {
        std::vector<unsigned long long> t(512);
        CB2_CUDA(cudaMemcpy(t.data(), trace_.p, t.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        const unsigned long long t0 = t[0];
        if (fused_trunk_)
            std::fprintf(stderr, "trunk trace (cycles since the stem's inputs; n=%u): layer: issuer has k-chunk 0 / 1 / last, last MMA issued | epilogue sees the accumulator, "
                                 "first chunk signalled by warp set 0 / 1, last chunk signalled\n", n);
        else
        std::fprintf(stderr, "trunk trace (cycles since layer 0 issue; n=%u): layer: inputs_ready mma_issued | acc_full ld_done stored fenced arrived\n", n);
        for (uint32_t l = 0; l <= 1 + 2 * d_.r && l < 64; ++l) {
            std::fprintf(stderr, "  l%-2u:", l);
            for (int k = 0; k < (fused_trunk_ ? 8 : 7); ++k) std::fprintf(stderr, " %8lld", static_cast<long long>(t[l * 8 + k] - t0));
            std::fprintf(stderr, "\n");
        }
        std::fprintf(stderr, "issuer per (layer, first tile of group): arrive_at_wait inputs_ready issued\n");
        for (uint32_t l = 0; l < 4; ++l)
            for (uint32_t g0 = 0; g0 < 8; ++g0) {
                const unsigned long long* e = &t[128 + (l * 8 + g0) * 3];
                if (e[2] == 0) continue;
                std::fprintf(stderr, "  l%u t%u: %8lld %8lld %8lld\n", l, g0, static_cast<long long>(e[0] - t0), static_cast<long long>(e[1] - t0),
                             static_cast<long long>(e[2] - t0));
            }
    }
    if (trace_.p != nullptr && stage == 2 && std::getenv("CATTUS_B200_TRACE_HEADS")) {
        std::vector<unsigned long long> t(512);
        CB2_CUDA(cudaMemcpy(t.data(), trace_.p, t.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        const unsigned long long t0 = t[0];
        std::fprintf(stderr, "heads trace (cycles since entry; n=%u): past n check %lld, setup done %lld, acc full %lld, epilogue done %lld, exit %lld\n", n,
                     static_cast<long long>(t[1] - t0), static_cast<long long>(t[2] - t0), static_cast<long long>(t[3] - t0),
                     static_cast<long long>(t[4] - t0), static_cast<long long>(t[5] - t0));
        unsigned long long ns0 = ~0ull;
        for (int y = 0; y < 17; ++y)
            if (t[256 + 4 * y] != 0) ns0 = std::min(ns0, t[256 + 4 * y]);
        std::fprintf(stderr, "  CTA (value, then policy N tiles): entry ns, exit ns (since the first entry), cycles inside\n");
        for (int y = 0; y < 17; ++y)
            if (t[256 + 4 * y] != 0)
                std::fprintf(stderr, "  %2d: %6lld %6lld %8lld\n", y, static_cast<long long>(t[256 + 4 * y] - ns0), static_cast<long long>(t[256 + 4 * y + 2] - ns0),
                             static_cast<long long>(t[256 + 4 * y + 3] - t[256 + 4 * y + 1]));
        std::fprintf(stderr, "  k-block: stage free (producer) | arrives at wait, stage full (issuer)\n");
        for (int kb = 0; kb < 40; ++kb)
            if (t[8 + kb] != 0)
                std::fprintf(stderr, "  %2d: %8lld | %8lld %8lld\n", kb, static_cast<long long>(t[48 + kb] - t0), static_cast<long long>(t[88 + kb] - t0),
                             static_cast<long long>(t[8 + kb] - t0));
    }
    for (auto& x : ev) cudaEventDestroy(x);
    std::lock_guard<std::mutex> g(m_mu_);
    metrics_.kernel_launches += launched;
}

// stage 5: every iteration is ONE pass of the whole launch sequence (L2 flushed before it, not inside it) with an event
// after each stage, so the three durations [encode + trunk, heads, tail] add up to the pass: the heads read the trunk's
// output from L2 exactly as they do inside the graph.  ms_out holds 3 * iters values.
void Engine::time_stages_split(uint32_t n, uint32_t iters, float* ms_out) {
    if (n == 0 || n > max_batch_ || iters == 0) throw Error(CATTUS_B200_EINVAL, "time_stage: bad argument");
    CB2_CUDA(cudaSetDevice(device_));
    Lane& l = *lanes_[0];
    if (flush_.p == nullptr) flush_.alloc(256ull << 20);
    std::vector<Op>& ops = ops_for(l, bucket_for(n), false);
    std::vector<cudaEvent_t> ev(4 * iters);
    for (auto& x : ev) CB2_CUDA(cudaEventCreate(&x));
    for (uint32_t it = 0; it < iters; ++it) {
        CB2_CUDA(cudaMemsetAsync(flush_.p, static_cast<int>(it & 0xFF), flush_.bytes, l.stream));
        CB2_CUDA(cudaEventRecord(ev[4 * it], l.stream));
        int group = 0;  // 0: stages 0-1, 1: stage 2, 2: stage 3
        for (const Op& op : ops) {
            const int g = op.stage <= 1 ? 0 : op.stage - 1;
            while (group < g) CB2_CUDA(cudaEventRecord(ev[4 * it + ++group], l.stream));
            op.launch(l.stream);
        }
        while (group < 3) CB2_CUDA(cudaEventRecord(ev[4 * it + ++group], l.stream));
    }
    cudaError_t se = cudaStreamSynchronize(l.stream);
    if (se != cudaSuccess) throw_device_error("time_stage", se);
    for (uint32_t it = 0; it < iters; ++it)
        for (int g = 0; g < 3; ++g) CB2_CUDA(cudaEventElapsedTime(&ms_out[3 * it + g], ev[4 * it + g], ev[4 * it + g + 1]));
    for (auto& x : ev) cudaEventDestroy(x);
    std::lock_guard<std::mutex> g(m_mu_);
    metrics_.kernel_launches += static_cast<uint64_t>(iters) * ops.size();
}

// Sustained throughput: n_batches DISTINCT resident batches (one per lane), `iters` graph replays rotating over them back
// to back on one stream, one pair of events around the lot.  No L2 flush: the rotation itself keeps the inputs cold and the
// weights warm, as in production.
void Engine::time_sustained(const uint64_t* planes, const uint8_t* legal, uint32_t n, uint32_t n_batches, uint32_t iters, float* total_ms) {
    if (n == 0 || n > max_batch_ || n_batches == 0 || n_batches > lanes_.size() || iters == 0 || !planes || !total_ms)
        throw Error(CATTUS_B200_EINVAL, "time_sustained: bad argument (n_batches must not exceed n_streams)");
    CB2_CUDA(cudaSetDevice(device_));
    std::vector<Lane*> held;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    try {
        for (uint32_t k = 0; k < n_batches; ++k) held.push_back(&acquire_lane());
        const size_t plane_words = static_cast<size_t>(rec_.planes) * rec_.wpp;
        const size_t bm = d_.bitmap_bytes();
        for (uint32_t k = 0; k < n_batches; ++k) {
            Lane& l = *held[k];
            uint32_t total = 0;
            for (uint32_t i = 0; i < n; ++i) {
                const size_t b = static_cast<size_t>(k) * n + i;
                total += pack_record(l.h_in + kRecs0 + static_cast<size_t>(i) * rec_.rec_bytes, planes + b * plane_words, legal ? legal + b * bm : nullptr, total);
            }
            *reinterpret_cast<uint32_t*>(l.h_in) = n;
            CB2_CUDA(cudaMemcpyAsync(l.d_in.p, l.h_in, 16 + static_cast<size_t>(n) * rec_.rec_bytes, cudaMemcpyHostToDevice, l.stream));
            run_bucket(l, bucket_for(n), l.stream, true, false);  // builds / warms the lane's graph
            CB2_CUDA(cudaStreamSynchronize(l.stream));
        }
        cudaStream_t st = held[0]->stream;
        CB2_CUDA(cudaEventCreate(&e0));
        CB2_CUDA(cudaEventCreate(&e1));
        CB2_CUDA(cudaEventRecord(e0, st));
        for (uint32_t it = 0; it < iters; ++it) run_bucket(*held[it % n_batches], bucket_for(n), st, true, false);
        CB2_CUDA(cudaEventRecord(e1, st));
        cudaError_t se = cudaStreamSynchronize(st);
        if (se != cudaSuccess) throw_device_error("time_sustained", se);
        CB2_CUDA(cudaEventElapsedTime(total_ms, e0, e1));
        std::lock_guard<std::mutex> g(m_mu_);
        metrics_.kernel_launches += static_cast<uint64_t>(iters + n_batches) * kernels_per_batch_;
    } catch (...) {
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        for (Lane* l : held) release_lane(*l);
        throw;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    for (Lane* l : held) release_lane(*l);
}

void Engine::get_info(cattus_b200_info* info) const {
    std::memset(info, 0, sizeof(*info));
    info->game = d_.game;
    info->board_size = d_.s;
    info->planes = d_.c_in;
    info->moves = d_.moves;
    info->filters = d_.f;
    info->blocks = d_.r;
    info->value_channels = d_.vh;
    info->policy_channels = d_.ph;
    info->words_per_plane = d_.wpp();
    info->legal_bitmap_bytes = d_.bitmap_bytes();
    info->max_batch = max_batch_;
    info->n_streams = static_cast<uint32_t>(lanes_.size());
    info->precision = precision_;
    info->sm_count = static_cast<uint32_t>(sm_count_);
    info->kernels_per_batch = kernels_per_batch_;
    info->trunk_path = simple_ ? CATTUS_B200_TRUNK_DENSE : fused_trunk_ ? CATTUS_B200_TRUNK_FUSED : small_trunk_ ? CATTUS_B200_TRUNK_SMALL : precision_ == CATTUS_B200_PRECISION_FP32_CHECK ? CATTUS_B200_TRUNK_FP32 : CATTUS_B200_TRUNK_PER_LAYER;
}

void Engine::get_metrics(cattus_b200_metrics* m) const {
    std::lock_guard<std::mutex> g(m_mu_);
    *m = metrics_;
}

}  // namespace cb2

// ================================================================================================ C ABI
struct cattus_b200 {
    cb2::Engine* engine;
};

#include "dsearch.cuh"

static thread_local std::string g_last_error;

template <class F>
static int guarded(F&& f) {
    try {
        f();
        g_last_error.clear();
        return CATTUS_B200_OK;
    } catch (const cb2::Error& e) {
        g_last_error = e.what();
        return e.code;
    } catch (const std::bad_alloc&) {
        g_last_error = "out of host memory";
        return CATTUS_B200_ENOMEM;
    } catch (const std::exception& e) {
        g_last_error = e.what();
        return CATTUS_B200_EINVAL;
    } catch (...) {
        g_last_error = "unknown error";
        return CATTUS_B200_EINVAL;
    }
}

// a session call: SpError (the host driver's) carries its own code
template <class F>
static int session_guarded(F&& f) {
    return guarded([&] {
        try {
            f();
        } catch (const sp::SpError& e) {
            throw cb2::Error(e.code ? e.code : CATTUS_B200_EINVAL, e.msg);
        }
    });
}

extern "C" {

int cattus_b200_create_from_memory(const cattus_b200_desc* desc, const void* blob, size_t blob_bytes, cattus_b200_t** out) {
    return guarded([&] {
        if (!desc || !out) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        if (desc->struct_size != sizeof(cattus_b200_desc)) throw cb2::Error(CATTUS_B200_EINVAL, "descriptor struct_size mismatch (ABI version?)");
        *out = nullptr;
        std::unique_ptr<cb2::Engine> e(new cb2::Engine(*desc, blob, blob_bytes));
        *out = new cattus_b200{e.release()};
    });
}

int cattus_b200_create(const cattus_b200_desc* desc, cattus_b200_t** out) {
    return guarded([&] {
        if (!desc || !out) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        if (!desc->weights_path) throw cb2::Error(CATTUS_B200_EINVAL, "weights_path is NULL");
        std::ifstream f(desc->weights_path, std::ios::binary);
        if (!f) throw cb2::Error(CATTUS_B200_EINVAL, std::string("cannot open weight blob ") + desc->weights_path);
        std::vector<char> bytes((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
        cattus_b200_t* h = nullptr;
        const int rc = cattus_b200_create_from_memory(desc, bytes.data(), bytes.size(), &h);
        if (rc != CATTUS_B200_OK) throw cb2::Error(rc, g_last_error);
        *out = h;
    });
}

void cattus_b200_destroy(cattus_b200_t* h) {
    if (!h) return;
    delete h->engine;
    delete h;
}

int cattus_b200_get_info(const cattus_b200_t* h, cattus_b200_info* info) {
    return guarded([&] {
        if (!h || !info) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        h->engine->get_info(info);
    });
}

int cattus_b200_eval(cattus_b200_t* h, const uint64_t* planes, const uint8_t* legal_bitmap, float* probs_out, uint32_t probs_cap,
                     uint32_t* n_probs, float* value_out) {
    return guarded([&] {
        if (!h || !planes || !probs_out || !n_probs || !value_out) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        cb2::LeafRequest req;
        req.probs_out = probs_out;
        req.probs_cap = probs_cap;
        req.n_probs = n_probs;
        req.value_out = value_out;
        h->engine->eval_leaf(planes, legal_bitmap, &req);
    });
}

int cattus_b200_eval_batch(cattus_b200_t* h, const uint64_t* planes, const uint8_t* legal_bitmaps, uint32_t n, float* probs_out,
                           size_t probs_cap, uint32_t* prob_offsets, float* values_out) {
    return guarded([&] {
        if (!h) throw cb2::Error(CATTUS_B200_EINVAL, "null handle");
        h->engine->eval_batch(planes, legal_bitmaps, n, probs_out, probs_cap, prob_offsets, values_out);
    });
}

int cattus_b200_eval_batch_submit(cattus_b200_t* h, const uint64_t* planes, const uint8_t* legal_bitmaps, uint32_t n, int block, int32_t* ticket) {
    return guarded([&] {
        if (!h || !ticket) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        *ticket = h->engine->eval_batch_submit(planes, legal_bitmaps, n, block != 0);
    });
}

int cattus_b200_eval_batch_wait(cattus_b200_t* h, int32_t ticket, float* probs_out, size_t probs_cap, uint32_t* prob_offsets, float* values_out) {
    return guarded([&] {
        if (!h) throw cb2::Error(CATTUS_B200_EINVAL, "null handle");
        h->engine->eval_batch_wait(ticket, probs_out, probs_cap, prob_offsets, values_out);
    });
}

int cattus_b200_encode(cattus_b200_t* h, const uint64_t* planes, uint32_t n, uint32_t batch_size, float* nchw_out) {
    return guarded([&] {
        if (!h || !planes || !nchw_out) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        h->engine->encode(planes, n, batch_size, nchw_out);
    });
}

int cattus_b200_run_dense(cattus_b200_t* h, const float* nchw, uint32_t n, float* logits_out, float* values_out) {
    return guarded([&] {
        if (!h) throw cb2::Error(CATTUS_B200_EINVAL, "null handle");
        h->engine->run_dense(nchw, n, logits_out, values_out);
    });
}

int cattus_b200_resident_upload(cattus_b200_t* h, const uint64_t* planes, const uint8_t* legal_bitmaps, uint32_t n) {
    return guarded([&] {
        if (!h || !planes) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        h->engine->resident_upload(planes, legal_bitmaps, n);
    });
}

int cattus_b200_eval_resident(cattus_b200_t* h, uint32_t n, void* stream) {
    return guarded([&] {
        if (!h) throw cb2::Error(CATTUS_B200_EINVAL, "null handle");
        h->engine->eval_resident(n, static_cast<cudaStream_t>(stream));
    });
}

int cattus_b200_resident_download(cattus_b200_t* h, uint32_t n, float* probs_out, size_t probs_cap, uint32_t* prob_offsets,
                                  float* values_out) {
    return guarded([&] {
        if (!h || !probs_out || !prob_offsets || !values_out) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        h->engine->resident_download(n, probs_out, probs_cap, prob_offsets, values_out);
    });
}

int cattus_b200_time_stage(cattus_b200_t* h, uint32_t stage, uint32_t n, uint32_t iters, float* ms_out) {
    return guarded([&] {
        if (!h || !ms_out) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        h->engine->time_stage(stage, n, iters, ms_out);
    });
}

int cattus_b200_time_sustained(cattus_b200_t* h, const uint64_t* planes, const uint8_t* legal_bitmaps, uint32_t n, uint32_t n_batches, uint32_t iters,
                               float* total_ms) {
    return guarded([&] {
        if (!h) throw cb2::Error(CATTUS_B200_EINVAL, "null handle");
        h->engine->time_sustained(planes, legal_bitmaps, n, n_batches, iters, total_ms);
    });
}

int cattus_b200_get_metrics(const cattus_b200_t* h, cattus_b200_metrics* out) {
    return guarded([&] {
        if (!h || !out) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        h->engine->get_metrics(out);
    });
}

// ---------------------------------------------------------------- batched analysis (include/cattus_b200_analysis.h)
struct cattus_b200_analysis {
    std::vector<ds::AnalysisResult> res;
};

int cattus_b200_analyse(cattus_b200_t* model, const cattus_b200_selfplay_cfg* cfg, uint32_t n, const char* const* fens, const uint16_t* moves,
                        const uint32_t* move_offsets, cattus_b200_analysis_t** out) {
    return guarded([&] {
        if (!cfg || !out) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        *out = nullptr;
        std::unique_ptr<cattus_b200_analysis> r(new cattus_b200_analysis());
        cb2::analyse_run(model, *cfg, 1, n, fens, moves, move_offsets, r->res);
        *out = r.release();
    });
}

int cattus_b200_analyse_opts(cattus_b200_t* model, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_analysis_opts* opts, uint32_t n,
                             const char* const* fens, const uint16_t* moves, const uint32_t* move_offsets, cattus_b200_analysis_t** out) {
    return guarded([&] {
        if (!cfg || !out) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        *out = nullptr;
        uint32_t search_batch = 1;
        try {
            search_batch = ds::analysis_search_batch(opts);
        } catch (const sp::SpError& e) {
            throw cb2::Error(e.code, e.msg);
        }
        std::unique_ptr<cattus_b200_analysis> r(new cattus_b200_analysis());
        cb2::analyse_run(model, *cfg, search_batch, n, fens, moves, move_offsets, r->res);
        *out = r.release();
    });
}

int cattus_b200_analysis_count(const cattus_b200_analysis_t* r, uint32_t* n) {
    if (!r || !n) return CATTUS_B200_EINVAL;
    *n = static_cast<uint32_t>(r->res.size());
    return CATTUS_B200_OK;
}
int cattus_b200_analysis_get(const cattus_b200_analysis_t* r, uint32_t k, cattus_b200_analysis_position* out) {
    return r ? ds::analysis_get(r->res, k, out) : CATTUS_B200_EINVAL;
}
int cattus_b200_analysis_children(const cattus_b200_analysis_t* r, uint32_t k, uint16_t* moves, uint32_t* visits, float* w, float* priors,
                                  uint32_t cap) {
    return r ? ds::analysis_children(r->res, k, moves, visits, w, priors, cap) : CATTUS_B200_EINVAL;
}
int cattus_b200_analysis_pv(const cattus_b200_analysis_t* r, uint32_t k, uint16_t* pv, uint32_t cap) {
    return r ? ds::analysis_pv(r->res, k, pv, cap) : CATTUS_B200_EINVAL;
}
int cattus_b200_analysis_batches(const cattus_b200_analysis_t* r, uint32_t k, uint32_t* minibatches, uint32_t* collisions) {
    return r ? ds::analysis_batches(r->res, k, minibatches, collisions) : CATTUS_B200_EINVAL;
}
void cattus_b200_analysis_free(cattus_b200_analysis_t* r) { delete r; }

// ---------------------------------------------------------------- persistent search sessions (include/cattus_b200_session.h)
struct cattus_b200_session {
    std::unique_ptr<ds::SessionBase> s;
};

int cattus_b200_session_create(cattus_b200_t* model, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_session_opts* opts,
                               cattus_b200_session_t** out) {
    return session_guarded([&] {
        if (!cfg || !out) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        *out = nullptr;
        std::unique_ptr<cattus_b200_session> r(new cattus_b200_session());
        r->s = cb2::session_create(model, *cfg, opts);
        *out = r.release();
    });
}
int cattus_b200_session_set_position(cattus_b200_session_t* s, const char* fen, const uint16_t* moves, uint32_t n) {
    return session_guarded([&] {
        if (!s) throw cb2::Error(CATTUS_B200_EINVAL, "null session");
        s->s->set_position(fen, moves, n);
    });
}
int cattus_b200_session_new_game(cattus_b200_session_t* s) {
    return session_guarded([&] {
        if (!s) throw cb2::Error(CATTUS_B200_EINVAL, "null session");
        s->s->new_game();
    });
}
int cattus_b200_session_go(cattus_b200_session_t* s, const cattus_b200_session_limits* limits) {
    return session_guarded([&] {
        if (!s || !limits) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        s->s->go(*limits);
    });
}
int cattus_b200_session_stop(cattus_b200_session_t* s) {
    return session_guarded([&] {
        if (!s) throw cb2::Error(CATTUS_B200_EINVAL, "null session");
        s->s->stop();
    });
}
int cattus_b200_session_info(cattus_b200_session_t* s, cattus_b200_session_snapshot* out) {
    return session_guarded([&] {
        if (!s || !out) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        if (out->struct_size != sizeof(cattus_b200_session_snapshot)) throw cb2::Error(CATTUS_B200_EINVAL, "session snapshot struct_size mismatch");
        s->s->info(*out);
    });
}
int cattus_b200_session_wait(cattus_b200_session_t* s, uint32_t timeout_ms, cattus_b200_analysis_t** result) {
    bool done = false;
    std::unique_ptr<cattus_b200_analysis> r(new cattus_b200_analysis());
    const int rc = session_guarded([&] {
        if (!s || !result) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        *result = nullptr;
        done = s->s->wait(timeout_ms, r->res);
    });
    if (rc != CATTUS_B200_OK) return rc;
    if (!done) return CATTUS_B200_SESSION_RUNNING;
    *result = r.release();
    return CATTUS_B200_OK;
}
int cattus_b200_session_result_stats(const cattus_b200_analysis_t* r, cattus_b200_session_stats* out) {
    return r ? ds::session_stats(r->res, out) : CATTUS_B200_EINVAL;
}
void cattus_b200_session_destroy(cattus_b200_session_t* s) { delete s; }

// ---------------------------------------------------------------- match play from openings (include/cattus_b200_match.h)
struct cattus_b200_match {
    ds::MatchResult res;
};

int cattus_b200_match_run(cattus_b200_t* model_a, cattus_b200_t* model_b, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_match_side* side_b,
                          uint32_t n, const char* const* fens, const uint16_t* moves, const uint32_t* move_offsets, cattus_b200_match_t** out) {
    return guarded([&] {
        if (!cfg || !out) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        *out = nullptr;
        const uint32_t one[2] = {1, 1};
        std::unique_ptr<cattus_b200_match> r(new cattus_b200_match());
        cb2::match_run(model_a, model_b, *cfg, side_b, one, n, fens, moves, move_offsets, r->res);
        *out = r.release();
    });
}

int cattus_b200_match_run_opts(cattus_b200_t* model_a, cattus_b200_t* model_b, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_match_side* side_b,
                               const cattus_b200_match_opts* opts, uint32_t n, const char* const* fens, const uint16_t* moves,
                               const uint32_t* move_offsets, cattus_b200_match_t** out) {
    return guarded([&] {
        if (!cfg || !out) throw cb2::Error(CATTUS_B200_EINVAL, "null argument");
        *out = nullptr;
        uint32_t search_batch[2];
        try {
            ds::match_search_batch(opts, search_batch);
        } catch (const sp::SpError& e) {
            throw cb2::Error(e.code, e.msg);
        }
        std::unique_ptr<cattus_b200_match> r(new cattus_b200_match());
        cb2::match_run(model_a, model_b, *cfg, side_b, search_batch, n, fens, moves, move_offsets, r->res);
        *out = r.release();
    });
}
int cattus_b200_match_batches(const cattus_b200_match_t* r, uint32_t side, uint64_t* minibatches, uint64_t* collisions) {
    return r ? ds::match_batches(r->res, side, minibatches, collisions) : CATTUS_B200_EINVAL;
}

int cattus_b200_match_summary_get(const cattus_b200_match_t* r, cattus_b200_match_summary* out) {
    return r ? ds::match_summary(r->res, out) : CATTUS_B200_EINVAL;
}
int cattus_b200_match_opening_status(const cattus_b200_match_t* r, uint32_t k, uint32_t* status) {
    return r ? ds::match_opening_status(r->res, k, status) : CATTUS_B200_EINVAL;
}
int cattus_b200_match_game_get(const cattus_b200_match_t* r, uint32_t k, cattus_b200_match_game* out) {
    return r ? ds::match_game(r->res, k, out) : CATTUS_B200_EINVAL;
}
int cattus_b200_match_game_moves(const cattus_b200_match_t* r, uint32_t k, uint16_t* moves, uint32_t cap) {
    return r ? ds::match_game_moves(r->res, k, moves, cap) : CATTUS_B200_EINVAL;
}
void cattus_b200_match_free(cattus_b200_match_t* r) { delete r; }

const char* cattus_b200_last_error(void) { return g_last_error.c_str(); }
uint32_t cattus_b200_abi_version(void) { return CATTUS_B200_ABI_VERSION; }

}  // extern "C"
