// trunk_fused: the whole conv trunk of ConvNetV1 (stem + R residual blocks, training/cattus_train/net_utils.py:60-65,
// :23-42) for 8x8 boards and 128 filters in ONE persistent kernel, including the board -> feature-plane encoding
// (engine/src/net/mod.rs:121-156) of its input.
//
// Why it can be one kernel: a 3x3 "same" convolution never mixes two boards, so a CTA that owns a set of boards can
// carry them through all 1 + 2R layers without ever talking to another CTA.  Activations stay in shared memory as
// bf16 for the whole trunk; only the packed bitboards come in (144 B per board) and the final activations go out.
// The only streamed operand is the weights (295 KB per layer, identical for every CTA -> L2 hits).
//
// Work unit: a CTA pair (cluster of 2, tcgen05 cta_group::2) owns 8 boards per round: each CTA holds two 128-row
// tiles (2 boards each).  One tcgen05.mma covers M = 256 (one tile of each CTA), N = 128 output channels, K = 16
// input channels; each CTA stores only ITS 64 output channels of the weights (B operand is split across the pair),
// which halves both the weight bytes streamed per SM and the shared-memory operand reads per MMA.
//
// Shared-memory activation layout ("padded chunk planes", no swizzle, K-major UMMA core matrices):
//   for each 8-channel chunk c8 (16 B per cell) a plane of cells; cell(g, x) = (g + 2) * 9 + 1 + x where
//   g = 2 * y + j is the board row y of board j in {0,1} and x the file.  Every 8-cell segment is followed by one
//   zero cell and there are two zero segments above and below, so the input of tap (dy, dx) for output row
//   r = 8 g + x is simply cell(g, x) + 18 dy + dx: a 3x3 tap is the SAME descriptor with the start address moved
//   by (18 dy + dx) * 16 bytes.  8-row groups are 144 B apart (SBO), the two 8-channel halves of a K = 16 step are
//   one plane (162 cells, 2592 B) apart (LBO); consecutive planes share their zero margins.  Halo cells are zeroed
//   once and never written.  (Descriptor behaviour probed on hardware: tools/umma_probe.cu.)
//
// Pipeline per layer l, k-chunk kc (16 input channels), tile t:
//   producer (1 thread / CTA) : TMA of this CTA's half of the (l, kc) weight stage (9 taps x 2 KB) into a 3-slot ring;
//                               both CTAs' bytes are credited to the leader's "full" barrier
//   MMA issuer (1 thread, leader CTA): waits weights(l, kc) and "input chunk kc of tile t is written in both CTAs",
//                               issues 9 MMAs (one per tap) into accumulator (t, l & 1); commits free the ring slot
//                               (multicast to both CTAs) and, after the last k-chunk, publish the accumulator
//   epilogue (4 warps per tile): TMEM -> registers, + folded-BN bias (+ residual from smem) -> ReLU -> bf16 ->
//                               the other activation buffer, 16 channels at a time, signalling the leader's
//                               "input chunk ready" barrier after every 16 channels -- the k-chunk-outer MMA order
//                               lets layer l+1 start while layer l's epilogue is still draining.
// With two tiles per CTA the issuer alternates tiles, so one tile's epilogue hides behind the other tile's MMAs.
//
// The two 1x1 head convolutions (net_utils.py:69, :79) ride along as one extra "layer": a single weight stage holding
// all 8 k-chunks of the [VH + PH][128] matrix (N = VH + PH <= 64 split across the pair like every other layer), no
// taps, whose epilogue writes ReLU(bf16) straight into the FC kernels' A operands.  The 67 MB trunk output tensor
// (and the two launches that re-read it) of the unfused arrangement never exists.
//
// Widths (round 2): the kernel is a template over the filter count F in {64, 128, 256} -- the range the reference's chess
// config recommends (training/config/chess_dev.yaml:30-37).  What changes with F is geometry only (FtG<F> below): F / 16
// k-chunks per layer, F / 8 chunk planes per activation buffer, F / 2 output channels per CTA of the pair, F TMEM columns
// per accumulator.  F = 256 needs its activations (2 x 83 KB for ONE 128-row tile per CTA) and a weight ring in 227 KB, so
// its weight stages hold 3 taps of a k-chunk (12 KB, ring of 4) instead of all 9 (F <= 128: 9 taps, ring of 3), and it
// always runs one tile per CTA: layer l + 1's MMAs start on chunk 0 while layer l's epilogue is still writing chunk 1.., so
// the tensor pipe stays fed without a second tile as long as a layer's MMAs outlast its epilogue (they do: 144 MMAs of
// M256 x N256 x K16 against 16 epilogue chunks).
//
// FP8 (opt-in, CATTUS_B200_PRECISION_FP8): the element type E is the second template parameter.  With E = e4m3 a 16-byte
// cell holds 16 channels instead of 8, so the geometry carries over: a chunk plane holds 16 channels (F / 16 planes per
// buffer), a k-chunk is 32 channels (ONE tcgen05.mma.kind::f8f6f4 of K = 32 per tap, F / 32 k-chunks per layer, one for
// the stem), SBO / LBO / tap shift are unchanged, and a weight stage [tap][k-half 2][oc F / 2][ic 16] has the bf16 stage's
// bytes -- half the stages per layer.  Numerics (oracle/fp8.py: convnet_forward_fp8 implements the same): weights are
// quantised per output channel to amax -> 448 at load, the epilogue computes relu(acc * d_oc + bias_oc (+ residual)) in
// fp32 and writes the next layer's A operand as e4m3 (round to nearest even, satfinite).  The residual stream stays bf16:
// a tile's block input also lives in a compact [F / 8][128 rows][8] bf16 buffer R beside P and Q, which the stem and
// every conv2 epilogue write and conv2 adds.  Head-conv outputs are bf16 as in the bf16 kernel.
#pragma once
#include <cuda_fp8.h>

#include "kernels.cuh"
#include "ptx.cuh"

namespace cb2 {

constexpr int kFtThreads = 384;  // warp 0 producer, 1 MMA issuer, 2 TMEM allocator, 3 idle, 4..11 epilogue
constexpr int kFtSegCells = 9;
constexpr int kFtPlaneCells = 162;                             // (16 + 2) segments
constexpr int kFtCell0 = 19;                                   // cell(g = 0, x = 0)
constexpr int kFtLbo = kFtPlaneCells * 16;                     // 2592
constexpr int kFtSbo = kFtSegCells * 16;                       // 144

// Geometry of the F-filter variant with element type E (__nv_bfloat16 or __nv_fp8_e4m3).
template <int F, typename E>
struct FtG {
    static_assert(F == 64 || F == 128 || F == 256, "trunk_fused covers 64, 128 and 256 filters");
    static_assert(sizeof(E) == 2 || sizeof(E) == 1, "trunk_fused covers bf16 and e4m3");
    static constexpr bool kFp8 = sizeof(E) == 1;
    static constexpr int kCellCh = 16 / static_cast<int>(sizeof(E));   // channels per 16-byte cell = per chunk plane
    static constexpr int kKch = 2 * kCellCh;                            // channels per k-chunk (one MMA per tap: K = 16 bf16 / 32 e4m3)
    static constexpr int kKc = F / kKch;                                // k-chunks per layer
    static constexpr int kStemKc = 32 / kKch;                           // the stem's input is padded to 32 channels
    static constexpr int kBufBytes = (F / kCellCh - 1) * kFtLbo + 181 * 16;  // F / kCellCh chunk planes, margins shared (F = 128 bf16: 41776)
    static constexpr int kResBytes = kFp8 ? F * 128 * 2 : 0;            // FP8: bf16 residual copy R [F / 8][128 rows][8]
    static constexpr int kTileBytes = 2 * kBufBytes + kResBytes;        // per tile: P, Q (and R)
    static constexpr int kTilesMax = F <= 128 ? 2 : 1;                  // 128-row tiles per CTA
    static constexpr int kActBytes = kTilesMax * kTileBytes;
    static constexpr int kWOff = (kActBytes + 127) / 128 * 128;
    static constexpr int kNpc = F / 2;                                  // output channels per CTA of the pair
    static constexpr int kTapBytes = 2 * kNpc * 16;                     // one tap of one k-chunk: [2 halves][kNpc oc][16 B of ic]
    static constexpr int kTapsPerStage = F <= 128 ? 9 : 3;
    static constexpr int kSubStages = 9 / kTapsPerStage;                // weight stages per (layer, k-chunk)
    static constexpr int kWStage = kTapsPerStage * kTapBytes;           // F = 128: 18432
    static constexpr int kWStages = F <= 128 ? 3 : 4;                   // ring depth
    // One tile per CTA (small batches) leaves the second tile's two activation buffers unused: they become extra ring slots.
    // A lone CTA pair pulls its weights from L2 with ~1 us per TMA round trip; three stages in flight deliver one stage per
    // ~0.33 us, about what its 9 MMAs take (0.29 us), so every hiccup shows -- a deeper ring keeps the tensor pipe fed.
    static constexpr int kExtraOff = (kTileBytes + 127) / 128 * 128;
    static constexpr int kExtraStages = kTilesMax == 2 ? (kWOff - kExtraOff) / kWStage : 0;
    static constexpr int kWStagesMax = kWStages + kExtraStages;
    static constexpr int kBlockBytes = 9 * kTapBytes;                   // weight image bytes of one (layer, k-chunk, CTA rank)
    static constexpr int kHeadStages = kKc > 8 ? kKc / 8 : 1;           // the head convs' [k-chunk][2][nh / 2][16 B] matrix, 8 k-chunks per stage
    static constexpr int kHeadKcPerStage = kKc / kHeadStages;
    static constexpr int kBarOff = kWOff + kWStages * kWStage;
    static constexpr int kNumBars = 2 * kWStagesMax + kTilesMax * kKc + 2 * kTilesMax;  // w_full, w_empty, act_full[tile][kc], acc_full[tile][2]
    static constexpr int kSmemBytes = kBarOff + kNumBars * 8 + 16 + 128;
    static constexpr int kWRowsPerStage = kWStage / 256;                // weight image is a u8 [rows][256] tensor
    static constexpr int kWRowsPerBlock = kBlockBytes / 256;
    static_assert(kSmemBytes <= 227 * 1024, "trunk_fused: shared memory");
    static_assert(kHeadKcPerStage * 64 * 16 <= kWStage, "trunk_fused: head stage");
};

struct alignas(64) TrunkFusedParams {
    CUtensorMap tma_w;       // weight image, u8 [rows][256], box {256, 72}
    const uint8_t* recs;     // packed records (planes first)
    const uint32_t* n_ptr;   // number of valid positions
    const float* bias;       // [layers + 1][F] folded-BN bias (last row: the head convs)
    const float* scale;      // FP8 only: [layers + 1][F] per-output-channel weight dequantisation factor d_oc; bf16: nullptr
    __nv_bfloat16* out_v;    // [boards * 64][vhp]  ReLU(value head conv)
    __nv_bfloat16* out_p;    // [boards * 64][php]  ReLU(policy head conv)
    uint32_t* err;
    int rec_bytes;
    int planes;      // C_in <= 32
    int layers;      // 1 + 2R
    int num_rounds;  // ceil(boards / (4 * tiles))
    int tiles;       // 128-row tiles per CTA in use: 2 (8 boards per pair and round) or, for small batches, 1 (4 boards: half the MMAs per round)
    int vhp, php;    // padded head widths (multiples of 16, vhp + php <= 64)
    unsigned long long* dbg;  // optional [layer][8] clock64 trace of pair 0, round 0 (CATTUS_B200_TRACE_TRUNK=1), else nullptr
};

// first k-chunk block of layer l in the weight image (the stem has kStemKc k-chunks, every other layer kKc)
template <int F, typename E>
__host__ __device__ __forceinline__ int ft_block_base(int l) {
    return l == 0 ? 0 : FtG<F, E>::kStemKc + (l - 1) * FtG<F, E>::kKc;
}

template <int F, typename E>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kFtThreads, 1) trunk_fused_kernel(const __grid_constant__ TrunkFusedParams p) {
    using G = FtG<F, E>;
    constexpr int kKc = G::kKc;
    constexpr bool kFp8 = G::kFp8;
    constexpr uint32_t kErrBase = kFp8 ? 0x8000u : 0u;  // fault codes of the FP8 instantiations: 0x9100.. instead of 0x1100..
    const uint32_t kWS = p.tiles == 1 ? G::kWStagesMax : G::kWStages;  // ring depth in use (uniform over the cluster)
    extern __shared__ uint8_t ft_smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ft_smem_raw) + 127) & ~static_cast<uintptr_t>(127));
    uint8_t* act = smem;
    uint64_t* w_full = reinterpret_cast<uint64_t*>(smem + G::kBarOff);
    uint64_t* w_empty = w_full + G::kWStagesMax;
    uint64_t* act_full = w_empty + G::kWStagesMax;          // [tile * kKc + kc]
    uint64_t* acc_full = act_full + G::kTilesMax * kKc;     // [tile * 2 + parity]
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_full + 2 * G::kTilesMax);

    const uint32_t warp = threadIdx.x >> 5;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t rank = ptx::cluster_ctarank();
    const int pair = blockIdx.x >> 1;
    const int num_pairs = gridDim.x >> 1;
    const int n_valid = static_cast<int>(*p.n_ptr);
    // Rounds that hold at least one valid position: the launch is sized for the batch bucket, but a round of nothing but
    // padding is skipped (every thread of both CTAs derives the same bound, so the barrier phases stay in step).
    const int rounds = min(p.num_rounds, (n_valid + 4 * p.tiles - 1) / (4 * p.tiles));

    // ---- one-time setup: zero the activation planes (halo cells stay zero for the whole kernel), barriers, TMEM
    for (int i = threadIdx.x; i < G::kActBytes / 16; i += kFtThreads) reinterpret_cast<uint4*>(act)[i] = make_uint4(0, 0, 0, 0);
    if (warp == 0 && lane == 0) ptx::prefetch_tensormap(&p.tma_w);
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < G::kWStagesMax; ++s) {
            ptx::mbar_init(&w_full[s], 1);
            ptx::mbar_init(&w_empty[s], 1);
        }
        for (int i = 0; i < G::kTilesMax * kKc; ++i) ptx::mbar_init(&act_full[i], 8);  // 4 epilogue warps x 2 CTAs
        for (int i = 0; i < 2 * G::kTilesMax; ++i) ptx::mbar_init(&acc_full[i], 1);
        ptx::fence_barrier_init();
    }
    if (warp == 2) {
        ptx::tmem_alloc_pair(tmem_ptr, 512);
        ptx::tmem_relinquish_pair();
    }
    ptx::fence_proxy_async_smem();
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    // byte offset (from `smem`) of ring slot i: the ring proper, then the idle tile's activation buffers
    auto slot_off = [](uint32_t i) -> uint32_t {
        return i < static_cast<uint32_t>(G::kWStages) ? static_cast<uint32_t>(G::kWOff) + i * G::kWStage
                                                      : static_cast<uint32_t>(G::kExtraOff) + (i - G::kWStages) * G::kWStage;
    };

    if (warp == 0) {
        // ================================================================== weight producer (both CTAs)
        if (lane == 0) {
            uint32_t it = 0;
            auto load_stage = [&](int row) {
                const uint32_t slot = it % kWS, ph = (it / kWS) & 1;
                ptx::mbar_wait(&w_empty[slot], ph ^ 1, p.err, kErrBase + 0x1100 + slot);
                if (rank == 0) ptx::mbar_arrive_expect_tx(&w_full[slot], 2 * G::kWStage);
                ptx::tma_load_2d_pair(smem + slot_off(slot), &p.tma_w, ptx::mapa(ptx::smem_u32(&w_full[slot]), 0), 0, row);
                ++it;
            };
            for (int rd = pair; rd < rounds; rd += num_pairs) {
                for (int l = 0; l < p.layers; ++l) {
                    const int nkc = l == 0 ? G::kStemKc : kKc;
                    for (int kc = 0; kc < nkc; ++kc) {
                        const int block = (ft_block_base<F, E>(l) + kc) * 2 + static_cast<int>(rank);
                        for (int sub = 0; sub < G::kSubStages; ++sub) load_stage(block * G::kWRowsPerBlock + sub * G::kWRowsPerStage);
                    }
                }
                // the head convs: kHeadStages stages inside one image block per CTA rank
                const int hblock = ft_block_base<F, E>(p.layers) * 2 + static_cast<int>(rank);
                for (int hs = 0; hs < G::kHeadStages; ++hs) load_stage(hblock * G::kWRowsPerBlock + hs * G::kWRowsPerStage);
            }
            // tail: do not leave while the leader's commits may still arrive on our barriers
            for (uint32_t j = it; j < it + kWS; ++j) ptx::mbar_wait(&w_empty[j % kWS], ((j / kWS) & 1) ^ 1, p.err, kErrBase + 0x1200 + (j % kWS));
        }
        __syncwarp();
    } else if (warp == 1) {
        // ================================================================== MMA issuer (leader CTA only)
        // The WHOLE warp runs this loop (warp-uniform control flow and addresses, so the compiler keeps descriptors in
        // uniform registers); only the tcgen05 instructions themselves are issued by one elected lane.  An earlier
        // version that ran the loop inside `if (lane == 0)` spent ~25 SASS instructions per MMA converting registers
        // to uniform registers and was issue-bound at half the tensor-pipe rate (profiles/r01c).
        if (rank == 0) {
            const uint32_t idesc = kFp8 ? ptx::umma_idesc_e4m3(256, F) : ptx::umma_idesc_bf16(256, F);
            const uint64_t a_hi64 = ptx::umma_desc_none_hi(kFtLbo, kFtSbo);
            const uint64_t b_hi64 = ptx::umma_desc_none_hi(G::kNpc * 16, 128);
            const uint32_t a_hi = static_cast<uint32_t>(a_hi64 >> 32), a_lo_fixed = static_cast<uint32_t>(a_hi64);
            const uint32_t b_hi = static_cast<uint32_t>(b_hi64 >> 32), b_lo_fixed = static_cast<uint32_t>(b_hi64);
            const uint32_t act_addr = ptx::smem_u32(act);
            const uint32_t smem_addr = ptx::smem_u32(smem);
            const bool leader_lane = ptx::elect_one();
            uint32_t act_par = 0;
            uint32_t it = 0;
            const int nh = p.vhp + p.php;
            const uint32_t idesc_head = kFp8 ? ptx::umma_idesc_e4m3(256, static_cast<uint32_t>(nh)) : ptx::umma_idesc_bf16(256, static_cast<uint32_t>(nh));
            const uint64_t bh_hi64 = ptx::umma_desc_none_hi(static_cast<uint32_t>(nh / 2) * 16, 128);
            const uint32_t bh_hi = static_cast<uint32_t>(bh_hi64 >> 32), bh_lo_fixed = static_cast<uint32_t>(bh_hi64);
            for (int rd = pair; rd < rounds; rd += num_pairs) {
                for (int l = 0; l < p.layers; ++l) {
                    const int nkc = l == 0 ? G::kStemKc : kKc;
                    const int in_buf = (l & 1) ? 1 : 0;  // stem and conv2 read P (0), conv1 reads Q (1)
                    for (int kc = 0; kc < nkc; ++kc) {
#pragma unroll
                        for (int sub = 0; sub < G::kSubStages; ++sub, ++it) {
                            const uint32_t slot = it % kWS, ph = (it / kWS) & 1;
                            ptx::mbar_wait(&w_full[slot], ph, p.err, kErrBase + 0x2100 + slot);
                            const uint32_t b_lo0 = b_lo_fixed | ((smem_addr + slot_off(slot)) >> 4);
#pragma unroll
                            for (int t = 0; t < G::kTilesMax; ++t) {
                                if (t >= p.tiles) break;
                                const int bi = t * kKc + kc;
                                if (sub == 0) {
                                    ptx::mbar_wait(&act_full[bi], (act_par >> bi) & 1u, p.err, kErrBase + 0x2200 + bi);
                                    act_par ^= 1u << bi;
                                }
                                ptx::tc_fence_after();
                                if (p.dbg != nullptr && pair == 0 && rd == 0 && t == 0 && sub == 0 && lane == 0 && (kc == 0 || kc == 1 || kc == nkc - 1))
                                    p.dbg[l * 8 + (kc == 0 ? 0 : kc == 1 ? 1 : 2)] = clock64();  // inputs of k-chunk 0 / 1 / last are there
                                const uint32_t a_lo0 = a_lo_fixed | ((act_addr + t * G::kTileBytes + in_buf * G::kBufBytes + (2 * kc) * kFtLbo + kFtCell0 * 16) >> 4);
                                const uint32_t d = tmem_base + static_cast<uint32_t>((t * 2 + (l & 1)) * F);
                                if (leader_lane) {
#pragma unroll
                                    for (int ts = 0; ts < G::kTapsPerStage; ++ts) {
                                        const int tap = sub * G::kTapsPerStage + ts;
                                        const int shift16 = 18 * (tap / 3 - 1) + (tap % 3 - 1);  // in 16-byte units
                                        if constexpr (kFp8)
                                            ptx::umma_f8_ss_pair_lohi(d, a_lo0 + shift16, a_hi, b_lo0 + ts * (G::kTapBytes / 16), b_hi, idesc, (kc | tap) != 0);
                                        else
                                            ptx::umma_bf16_ss_pair_lohi(d, a_lo0 + shift16, a_hi, b_lo0 + ts * (G::kTapBytes / 16), b_hi, idesc, (kc | tap) != 0);
                                    }
                                    if (kc == nkc - 1 && sub == G::kSubStages - 1) ptx::umma_commit_pair_multicast(&acc_full[t * 2 + (l & 1)], 3);
                                }
                                if (p.dbg != nullptr && pair == 0 && rd == 0 && t == 0 && lane == 0 && kc == nkc - 1 && sub == G::kSubStages - 1)
                                    p.dbg[l * 8 + 3] = clock64();  // last MMA of the layer issued
                            }
                            if (leader_lane) ptx::umma_commit_pair_multicast(&w_empty[slot], 3);
                            __syncwarp();
                        }
                    }
                }
                // ---- head convs: kKc k-chunks, no taps, N = vhp + php, input = Q (the last conv2 wrote it), accumulator parity 1
                for (int hs = 0; hs < G::kHeadStages; ++hs, ++it) {
                    const uint32_t slot = it % kWS, ph = (it / kWS) & 1;
                    ptx::mbar_wait(&w_full[slot], ph, p.err, kErrBase + 0x2100 + slot);
                    const uint32_t b_lo0 = bh_lo_fixed | ((smem_addr + slot_off(slot)) >> 4);
#pragma unroll
                    for (int t = 0; t < G::kTilesMax; ++t) {
                        if (t >= p.tiles) break;
                        const uint32_t d = tmem_base + static_cast<uint32_t>((t * 2 + 1) * F);
                        for (int k8 = 0; k8 < G::kHeadKcPerStage; ++k8) {
                            const int kc = hs * G::kHeadKcPerStage + k8;
                            const int bi = t * kKc + kc;
                            ptx::mbar_wait(&act_full[bi], (act_par >> bi) & 1u, p.err, kErrBase + 0x2300 + bi);
                            act_par ^= 1u << bi;
                            ptx::tc_fence_after();
                            const uint32_t a_lo = a_lo_fixed | ((act_addr + t * G::kTileBytes + G::kBufBytes + (2 * kc) * kFtLbo + kFtCell0 * 16) >> 4);
                            if (leader_lane) {
                                if constexpr (kFp8)
                                    ptx::umma_f8_ss_pair_lohi(d, a_lo, a_hi, b_lo0 + k8 * (nh / 2) * 2, bh_hi, idesc_head, kc != 0);
                                else
                                    ptx::umma_bf16_ss_pair_lohi(d, a_lo, a_hi, b_lo0 + k8 * (nh / 2) * 2, bh_hi, idesc_head, kc != 0);
                            }
                        }
                        if (leader_lane && hs == G::kHeadStages - 1) ptx::umma_commit_pair_multicast(&acc_full[t * 2 + 1], 3);
                    }
                    if (leader_lane) ptx::umma_commit_pair_multicast(&w_empty[slot], 3);
                    __syncwarp();
                }
            }
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ================================================================== encode + epilogue (4 warps per tile)
        // With ONE tile per CTA (small batches; F = 256 always) the second set of four warps would idle: it takes the odd
        // 16-channel chunks of tile 0 instead, so a layer's epilogue -- what the next layer's MMAs wait for -- takes half the
        // time.  Every chunk is still written and signalled by exactly four warps per CTA (one per TMEM lane quarter).
        const int wset = static_cast<int>(warp - 4) >> 2;
        const bool split = p.tiles == 1;
        const int t = split ? 0 : wset;
        const int kc0 = split ? wset : 0, kcs = split ? 2 : 1;
        const uint32_t q = warp & 3;  // TMEM lane quarter this warp may access
        const int r = static_cast<int>(q * 32 + lane);
        const int g = r >> 3, x = r & 7;
        const int j = g & 1, y = g >> 1;
        const int cell = y * 8 + x;
        const int pcell = kFtCell0 + g * kFtSegCells + x;
        uint8_t* bufP = act + t * G::kTileBytes + pcell * 16;
        uint8_t* bufQ = act + t * G::kTileBytes + G::kBufBytes + pcell * 16;
        uint8_t* bufR = act + t * G::kTileBytes + 2 * G::kBufBytes + r * 16;  // FP8: row r of R, 8-channel chunk c8 at + c8 * 2048
        const uint32_t leader_act = ptx::mapa(ptx::smem_u32(&act_full[t * kKc]), 0);
        const uint32_t tmem_row = tmem_base + ((q * 32u) << 16) + static_cast<uint32_t>(t * 2 * F);
        uint32_t acc_par = 0;
        for (int rd = pair; rd < rounds; rd += num_pairs) {
            const int board = ((rd * p.tiles + t) * 2 + static_cast<int>(rank)) * 2 + j;  // tile-major: a 1-tile round is boards 4 rd .. 4 rd + 3
            const bool valid = board < n_valid;
            // ---- planes_to_tensor for my cell: channels 0..31 of the stem input (planes >= C_in are zero)
            if (!split || wset == 0) {
                if constexpr (kFp8) {
                    uint32_t w[8];  // 32 channels, one e4m3 byte each (1.0 = 0x38)
#pragma unroll
                    for (int i = 0; i < 8; ++i) w[i] = 0;
                    if (valid) {
                        const uint64_t* pl = reinterpret_cast<const uint64_t*>(p.recs + static_cast<size_t>(board) * p.rec_bytes);
#pragma unroll
                        for (int c = 0; c < 32; ++c) {
                            if (c < p.planes && ((__ldg(pl + c) >> cell) & 1ull)) w[c >> 2] |= 0x38u << (8 * (c & 3));
                        }
                    }
#pragma unroll
                    for (int c16 = 0; c16 < 2; ++c16)
                        *reinterpret_cast<uint4*>(bufP + c16 * kFtLbo) = make_uint4(w[4 * c16], w[4 * c16 + 1], w[4 * c16 + 2], w[4 * c16 + 3]);
                } else {
                    uint32_t w[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) w[i] = 0;
                    if (valid) {
                        const uint64_t* pl = reinterpret_cast<const uint64_t*>(p.recs + static_cast<size_t>(board) * p.rec_bytes);
#pragma unroll
                        for (int c = 0; c < 32; ++c) {
                            if (c < p.planes && ((__ldg(pl + c) >> cell) & 1ull)) w[c >> 1] |= (c & 1) ? 0x3F800000u : 0x00003F80u;  // bf16 1.0
                        }
                    }
#pragma unroll
                    for (int c8 = 0; c8 < 4; ++c8)
                        *reinterpret_cast<uint4*>(bufP + c8 * kFtLbo) = make_uint4(w[4 * c8], w[4 * c8 + 1], w[4 * c8 + 2], w[4 * c8 + 3]);
                }
                ptx::tc_fence_before();  // orders my earlier tcgen05.ld of accumulator (t, 0) before the stem MMAs that overwrite it
                ptx::fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
#pragma unroll
                    for (int kc = 0; kc < G::kStemKc; ++kc) ptx::mbar_arrive_cluster(leader_act + kc * 8);
                }
            }
            for (int l = 0; l < p.layers; ++l) {
                // Last layer of this pair's last round: the head FC kernel may be staged now (it runs its prologue and then waits
                // for this whole grid).  Not earlier: staged CTAs hold their shared memory while they wait, and with many lanes
                // in flight they would take SMs away from the other lanes' trunks for the length of this kernel.
                if (l == p.layers - 1 && rd + num_pairs >= rounds && warp == 4 && lane == 0) ptx::grid_dep_launch();
                const int par = l & 1;
                const bool has_resid = l >= 2 && par == 0;  // conv2 of a block: + block input (Q), result back into Q
                uint8_t* outb = par ? bufP : bufQ;          // stem -> Q, conv1 -> P, conv2 -> Q
                const float4* bias4 = reinterpret_cast<const float4*>(p.bias + l * F);
                float4 bn[4];  // bias of the chunk about to be processed, fetched one chunk ahead (bf16)
                if constexpr (!kFp8) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) bn[i] = __ldg(bias4 + kc0 * 4 + i);
                }
                ptx::mbar_wait(&acc_full[t * 2 + par], (acc_par >> par) & 1u, p.err, kErrBase + 0x3100 + t * 2 + par);
                acc_par ^= 1u << par;
                ptx::tc_fence_after();
                const bool tr = p.dbg != nullptr && pair == 0 && rd == 0 && rank == 0 && t == 0 && q == 0 && lane == 0;
                if (tr && wset == 0) p.dbg[l * 8 + 4] = clock64();  // accumulator complete (seen by the epilogue)
#pragma unroll 1
                for (int kc = kc0; kc < kKc; kc += kcs) {
                  if constexpr (kFp8) {
                    // 32 channels: two halves of 16, each one e4m3 cell of the next layer's A (+ the bf16 residual copy)
                    const float4* b4 = bias4 + kc * 8;
                    const float4* s4 = reinterpret_cast<const float4*>(p.scale + l * F) + kc * 8;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        uint32_t raw[16];
                        ptx::tmem_ld_x16_issue(tmem_row + static_cast<uint32_t>(par * F + kc * 32 + h * 16), raw);
                        float4 bc[4], sc[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            bc[i] = __ldg(b4 + h * 4 + i);
                            sc[i] = __ldg(s4 + h * 4 + i);
                        }
                        ptx::tmem_ld_wait(raw);
                        float v[16];
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            v[4 * i + 0] = fmaf(__uint_as_float(raw[4 * i + 0]), sc[i].x, bc[i].x);
                            v[4 * i + 1] = fmaf(__uint_as_float(raw[4 * i + 1]), sc[i].y, bc[i].y);
                            v[4 * i + 2] = fmaf(__uint_as_float(raw[4 * i + 2]), sc[i].z, bc[i].z);
                            v[4 * i + 3] = fmaf(__uint_as_float(raw[4 * i + 3]), sc[i].w, bc[i].w);
                        }
                        uint8_t* rr8 = bufR + (kc * 4 + h * 2) * 2048;  // R chunks of channels kc * 32 + h * 16 + [0, 8), [8, 16)
                        if (has_resid) {
#pragma unroll
                            for (int c8 = 0; c8 < 2; ++c8) {
                                const uint4 rr = *reinterpret_cast<const uint4*>(rr8 + c8 * 2048);
                                const uint32_t rw[4] = {rr.x, rr.y, rr.z, rr.w};
#pragma unroll
                                for (int i = 0; i < 4; ++i) {
                                    const __nv_bfloat162 b2 = *reinterpret_cast<const __nv_bfloat162*>(&rw[i]);
                                    v[8 * c8 + 2 * i + 0] += __bfloat162float(b2.x);
                                    v[8 * c8 + 2 * i + 1] += __bfloat162float(b2.y);
                                }
                            }
                        }
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.0f);
                        if (par == 0) {  // stem / conv2: the output is the next block's input, whose bf16 copy conv2 will add
                            uint32_t o[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) {
                                const __nv_bfloat162 b2 = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
                                o[i] = *reinterpret_cast<const uint32_t*>(&b2);
                            }
                            *reinterpret_cast<uint4*>(rr8) = make_uint4(o[0], o[1], o[2], o[3]);
                            *reinterpret_cast<uint4*>(rr8 + 2048) = make_uint4(o[4], o[5], o[6], o[7]);
                        }
                        uint32_t e[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i) e[i] = ptx::cvt_e4m3x4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
                        *reinterpret_cast<uint4*>(outb + (2 * kc + h) * kFtLbo) = make_uint4(e[0], e[1], e[2], e[3]);
                    }
                  } else {
                    uint32_t raw[16];
                    ptx::tmem_ld_x16_issue(tmem_row + static_cast<uint32_t>(par * F + kc * 16), raw);
                    float4 bc[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) bc[i] = bn[i];
                    if (kc + kcs < kKc) {
#pragma unroll
                        for (int i = 0; i < 4; ++i) bn[i] = __ldg(bias4 + (kc + kcs) * 4 + i);
                    }
                    ptx::tmem_ld_wait(raw);
                    float v[16];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        v[4 * i + 0] = __uint_as_float(raw[4 * i + 0]) + bc[i].x;
                        v[4 * i + 1] = __uint_as_float(raw[4 * i + 1]) + bc[i].y;
                        v[4 * i + 2] = __uint_as_float(raw[4 * i + 2]) + bc[i].z;
                        v[4 * i + 3] = __uint_as_float(raw[4 * i + 3]) + bc[i].w;
                    }
                    if (has_resid) {
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            const uint4 rr = *reinterpret_cast<const uint4*>(bufQ + (2 * kc + h) * kFtLbo);
                            const uint32_t rw[4] = {rr.x, rr.y, rr.z, rr.w};
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                const __nv_bfloat162 b2 = *reinterpret_cast<const __nv_bfloat162*>(&rw[i]);
                                v[8 * h + 2 * i + 0] += __bfloat162float(b2.x);
                                v[8 * h + 2 * i + 1] += __bfloat162float(b2.y);
                            }
                        }
                    }
                    uint32_t o[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const __nv_bfloat162 b2 = __floats2bfloat162_rn(fmaxf(v[2 * i], 0.0f), fmaxf(v[2 * i + 1], 0.0f));
                        o[i] = *reinterpret_cast<const uint32_t*>(&b2);
                    }
                    *reinterpret_cast<uint4*>(outb + (2 * kc) * kFtLbo) = make_uint4(o[0], o[1], o[2], o[3]);
                    *reinterpret_cast<uint4*>(outb + (2 * kc + 1) * kFtLbo) = make_uint4(o[4], o[5], o[6], o[7]);
                  }
                    ptx::tc_fence_before();
                    ptx::fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive_cluster(leader_act + kc * 8);
                    if (tr && kc == kc0) p.dbg[l * 8 + 5 + (split ? wset : 0)] = clock64();  // first chunk of this warp set signalled
                    if (tr && kc + kcs >= kKc && (!split || wset == 1)) p.dbg[l * 8 + 7] = clock64();  // last chunk signalled
                }
            }
            // ---- both 1x1 head convolutions: accumulator (t, parity 1), columns [0, vhp) value, [vhp, vhp + php) policy
            {
                const float4* hb4 = reinterpret_cast<const float4*>(p.bias + p.layers * F);
                ptx::mbar_wait(&acc_full[t * 2 + 1], (acc_par >> 1) & 1u, p.err, kErrBase + 0x3200 + t);
                acc_par ^= 1u << 1;
                ptx::tc_fence_after();
                const size_t row = static_cast<size_t>(board) * 64 + cell;
                const int nh = p.vhp + p.php;
                for (int cb = 16 * kc0; cb < nh; cb += 16 * kcs) {
                    uint32_t raw[16];
                    ptx::tmem_ld_x16_issue(tmem_row + static_cast<uint32_t>(F + cb), raw);
                    float4 bc[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) bc[i] = __ldg(hb4 + cb / 4 + i);
                    if constexpr (kFp8) {
                        float4 sc[4];
                        const float4* hs4 = reinterpret_cast<const float4*>(p.scale + p.layers * F);
#pragma unroll
                        for (int i = 0; i < 4; ++i) sc[i] = __ldg(hs4 + cb / 4 + i);
                        ptx::tmem_ld_wait(raw);
#pragma unroll
                        for (int i = 0; i < 4; ++i) {  // dequantise: acc * d_oc; the bias is added below as in bf16
                            raw[4 * i + 0] = __float_as_uint(__uint_as_float(raw[4 * i + 0]) * sc[i].x);
                            raw[4 * i + 1] = __float_as_uint(__uint_as_float(raw[4 * i + 1]) * sc[i].y);
                            raw[4 * i + 2] = __float_as_uint(__uint_as_float(raw[4 * i + 2]) * sc[i].z);
                            raw[4 * i + 3] = __float_as_uint(__uint_as_float(raw[4 * i + 3]) * sc[i].w);
                        }
                    } else {
                        ptx::tmem_ld_wait(raw);
                    }
                    uint32_t o[8];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const __nv_bfloat162 a = __floats2bfloat162_rn(fmaxf(__uint_as_float(raw[4 * i + 0]) + bc[i].x, 0.0f),
                                                                       fmaxf(__uint_as_float(raw[4 * i + 1]) + bc[i].y, 0.0f));
                        const __nv_bfloat162 b = __floats2bfloat162_rn(fmaxf(__uint_as_float(raw[4 * i + 2]) + bc[i].z, 0.0f),
                                                                       fmaxf(__uint_as_float(raw[4 * i + 3]) + bc[i].w, 0.0f));
                        o[2 * i] = *reinterpret_cast<const uint32_t*>(&a);
                        o[2 * i + 1] = *reinterpret_cast<const uint32_t*>(&b);
                    }
                    if (valid) {
                        uint4* og = cb < p.vhp ? reinterpret_cast<uint4*>(p.out_v + row * p.vhp + cb) : reinterpret_cast<uint4*>(p.out_p + row * p.php + (cb - p.vhp));
                        og[0] = make_uint4(o[0], o[1], o[2], o[3]);
                        og[1] = make_uint4(o[4], o[5], o[6], o[7]);
                    }
                }
                ptx::tc_fence_before();
                // one tile, two warp sets: the next round's encode (set 0) lets the stem MMAs start, which in turn lets conv1
                // overwrite the parity-1 accumulator -- not before BOTH sets have read this round's head results out of it
                if (split) asm volatile("bar.sync 1, 256;" ::: "memory");
            }
        }
    }

    // ---- teardown: nobody leaves (or frees TMEM) before both CTAs are done
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync();
    if (warp == 2) ptx::tmem_dealloc_pair(tmem_base, 512);
}

}  // namespace cb2
