// CUDA side of the device-resident self-play: the three kernels that wrap dsearch_core.hpp (one warp per game), the
// captured "wave" graph  [zero counters] -> begin -> select -> evaluator kernels -> expand,  and the transport the host
// driver (dsearch_host.hpp) talks to.  Included at the end of engine.cu (single translation unit with the evaluator).
//
// Data path of one simulation, all in HBM: select writes the leaf's record into the evaluator lane's DEVICE input block
// (Engine::ResidentIo) and bumps its row counter; the evaluator's kernels read the row count from that block (as they
// always do) and leave values / probabilities in d_values / d_probs; expand reads them.  The host sees one small command
// block per wave going in (new games / chosen moves + Dirichlet samples) and the finished searches' root visit counts
// coming out through mapped pinned memory.
#pragma once

#include "dsearch_analysis.hpp"
#include "dsearch_api.hpp"
#include "dsearch_host.hpp"
#include "dsearch_match.hpp"
#include "dsearch_session.hpp"
#include "engine.hpp"

namespace cb2 {

#ifndef DS_SELECT_MIN_BLOCKS
#define DS_SELECT_MIN_BLOCKS 1
#endif
#ifndef DS_EXPAND_MIN_BLOCKS
#define DS_EXPAND_MIN_BLOCKS 1
#endif

template <class Rules>
__global__ void __launch_bounds__(128) ds_begin_kernel(ds::Params<Rules> p) {
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t* hdr = reinterpret_cast<const uint32_t*>(p.cmds);
    const uint32_t n_cmds = hdr[0], wave = hdr[1];
    if (warp >= n_cmds) return;
    decltype(auto) R = ds::RulesRef<Rules>::get(p.rules);
    ds::Core<Rules>::begin_slot(R, p, warp, wave);
}

// A session's begin (Core::begin_slot<true>, DESIGN.md section 17): its wave graph takes this one instead of ds_begin_kernel.
template <class Rules>
__global__ void __launch_bounds__(128) ds_begin_session_kernel(ds::Params<Rules> p) {
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t* hdr = reinterpret_cast<const uint32_t*>(p.cmds);
    const uint32_t n_cmds = hdr[0], wave = hdr[1];
    if (warp >= n_cmds) return;
    decltype(auto) R = ds::RulesRef<Rules>::get(p.rules);
    ds::Core<Rules>::template begin_slot<true>(R, p, warp, wave);
}

template <class Rules>
__global__ void __launch_bounds__(128, DS_SELECT_MIN_BLOCKS) ds_select_kernel(ds::Params<Rules> p) {
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (warp >= p.n_slots) return;
    const uint32_t wave = reinterpret_cast<const uint32_t*>(p.cmds)[1];
    decltype(auto) R = ds::RulesRef<Rules>::get(p.rules);
    ds::Core<Rules>::select_slot(R, p, warp, wave);
}

template <class Rules>
__global__ void __launch_bounds__(128, DS_EXPAND_MIN_BLOCKS) ds_expand_kernel(ds::Params<Rules> p) {
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (warp >= p.n_slots) return;
    const uint32_t wave = reinterpret_cast<const uint32_t*>(p.cmds)[1];
    decltype(auto) R = ds::RulesRef<Rules>::get(p.rules);
    ds::Core<Rules>::expand_slot(R, p, warp, wave);
}

// Minibatched search (a side with search_batch > 1, DESIGN.md sections 15 and 16): one warp per searched tree, captured
// in a wave graph of their own instead of select / expand.  The select kernel states its one block per SM: without it
// ptxas caps tic-tac-toe at 64 registers and spills, and hex 9-11 spill more.
template <class Rules>
__global__ void __launch_bounds__(128, 1) ds_select_batch_kernel(ds::Params<Rules> p) {
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (warp >= p.n_slots) return;
    const uint32_t wave = reinterpret_cast<const uint32_t*>(p.cmds)[1];
    decltype(auto) R = ds::RulesRef<Rules>::get(p.rules);
    ds::Core<Rules>::batch_select_slot(R, p, warp, wave);
}

template <class Rules>
__global__ void __launch_bounds__(128) ds_expand_batch_kernel(ds::Params<Rules> p) {
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (warp >= p.n_slots) return;
    const uint32_t wave = reinterpret_cast<const uint32_t*>(p.cmds)[1];
    decltype(auto) R = ds::RulesRef<Rules>::get(p.rules);
    ds::Core<Rules>::batch_expand_slot(R, p, warp, wave);
}

// One population of slots: its kernel parameters, streams, captured wave graph, command and status blocks, evaluator lanes
// and evaluation caches.  Two populations alternate waves on two streams (dsearch_host.hpp), so that one population's
// select / expand kernels run beside the other's evaluator kernels.
template <class Rules>
struct DsPopulation {
    ds::Params<Rules> p;
    Engine::ResidentIo io[2];
    cudaStream_t stream = nullptr, side = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
    cudaGraphExec_t graph = nullptr;
    void *d_cmds = nullptr, *d_status = nullptr, *d_cache_meta[2] = {nullptr, nullptr}, *d_cache_entries[2] = {nullptr, nullptr};
    void* d_roots = nullptr;  // root upload: root histories of the population's current wave
};

template <class Rules>
class DsCudaBackend {
  public:
    // `roots_cap` > 0 adds the per-wave root upload of kCmdSetRoot (analysis, matches from openings): up to that many
    // history positions per wave.  `search_batch` (optional) is each side's descents per minibatch: when one of them is
    // above 1 the waves run the minibatch kernels.  `analysis` (optional) switches the finished searches to the analysis
    // result layout.  `session_kwords` (optional, with analysis and search_batch > 1: a session, dsearch_session.hpp) makes
    // one slot whose tree buffers hold that many kwords (0: the most the tree address space allows), takes a free
    // evaluator lane or fails, and adds the session's control words and snapshot in mapped memory.  Without them
    // everything is the self-play arrangement.
    DsCudaBackend(const void* rules_blob, size_t rules_bytes, uint32_t max_children, Engine* e1, Engine* e2, const cattus_b200_selfplay_cfg& cfg,
                  const sp::Params params[2], uint32_t n_slots, uint32_t roots_cap = 0, const uint32_t* search_batch = nullptr,
                  const ds::AnalysisOpts* analysis = nullptr, const uint32_t* session_kwords = nullptr)
        : max_children_(max_children), n_slots_(n_slots), device_(e1->device()), session_(session_kwords != nullptr) {
        if (search_batch) {
            side_batch_[0] = std::max<uint32_t>(1, search_batch[0]);
            side_batch_[1] = std::max<uint32_t>(1, search_batch[1]);
            search_batch_ = std::max(side_batch_[0], side_batch_[1]);
        }
        eng_[0] = e1;
        eng_[1] = e2;
        n_evals_ = e2 ? 2 : 1;
        if (e2 && e2->device() != e1->device()) throw Error(CATTUS_B200_EINVAL, "device search: both models must live on the same device");
        CB2_CUDA(cudaSetDevice(e1->device()));
        depth_ = cfg.device_waves_in_flight ? std::min<uint32_t>(cfg.device_waves_in_flight, 8) : 2;
        n_bufs_ = depth_ + 1;
        wave_pop_.assign(n_bufs_, 0);
        const auto t0 = std::chrono::steady_clock::now();
        try {
            // evaluator lanes: one per population and evaluator; a second population needs a second free stream in every evaluator
            for (uint32_t e = 0; e < n_evals_; ++e) {
                pop_[0].io[e] = eng_[e]->resident_acquire(!session_);
                if (pop_[0].io[e].lane < 0)
                    throw Error(CATTUS_B200_EINVAL, "session: the model has no free evaluator lane; a session holds one for its lifetime, so create "
                                                    "the model with n_streams >= 2");
                if (search_batch_ > 1 && pop_[0].io[e].max_batch < static_cast<uint64_t>(n_slots) * search_batch_)
                    throw Error(CATTUS_B200_ERANGE, "device search: device_games (" + std::to_string(n_slots) + ") x search_batch (" +
                                                        std::to_string(search_batch_) + ") exceeds the evaluator's max_batch (" +
                                                        std::to_string(pop_[0].io[e].max_batch) + ")");
                if (pop_[0].io[e].max_batch < n_slots)
                    throw Error(CATTUS_B200_ERANGE, "device search: device_games (" + std::to_string(n_slots) + ") exceeds the evaluator's max_batch (" +
                                                        std::to_string(pop_[0].io[e].max_batch) + ")");
                if (pop_[0].io[e].moves < max_children && !Rules::kChess) throw Error(CATTUS_B200_EINVAL, "device search: the model's move count does not fit the game");
            }
            n_pops_ = 1;
            // Two populations taking waves in turn on two streams were measured and do NOT pay on a B200: the persistent trunk
            // kernels leave no room for the other population's select / expand blocks to run beside them, and half-size batches
            // are less efficient (hex5 64.1 M vs 64.4 M sims/s, hex7 30.0 M vs 37.1 M, chess 10x128 4.7 M vs 5.0 M).  Kept as an
            // experiment knob; the games are the same either way (tests/test_gpu_dsearch.py).
            if (n_slots >= 64 && depth_ >= 2 && search_batch_ == 1 && std::getenv("CATTUS_B200_DSEARCH_TWO_POPULATIONS")) {
                bool ok = true;
                for (uint32_t e = 0; e < n_evals_; ++e) {
                    pop_[1].io[e] = eng_[e]->resident_acquire(false);
                    ok = ok && pop_[1].io[e].lane >= 0;
                }
                if (ok) {
                    n_pops_ = 2;
                } else {
                    for (uint32_t e = 0; e < n_evals_; ++e)
                        if (pop_[1].io[e].lane >= 0) {
                            eng_[e]->resident_release(pop_[1].io[e].lane);
                            pop_[1].io[e].lane = -1;
                        }
                }
            }
            split_ = n_pops_ == 2 ? (n_slots + 1) / 2 : n_slots;

            using T = ds::TreeOps<Rules>;
            const uint32_t typ = Rules::kChess ? 48u : max_children;
            const uint64_t per_search = (static_cast<uint64_t>(std::max(params[0].sim_num, params[1].sim_num)) + 8u) * T::block_words(static_cast<int>(typ));
            uint64_t want = cfg.device_tree_kwords ? static_cast<uint64_t>(cfg.device_tree_kwords) * 1024u : 3u * per_search;
            size_t free_b = 0, total_b = 0;
            CB2_CUDA(cudaMemGetInfo(&free_b, &total_b));
            const uint64_t budget = static_cast<uint64_t>(static_cast<double>(free_b) * 0.7) / (static_cast<uint64_t>(n_slots) * 3u * 4u);
            if (!cfg.device_tree_kwords) want = std::min(want, budget);
            want &= ~static_cast<uint64_t>(3);
            if (session_) {  // sized by the session's options, not by sim_num (a session's searches have no fixed size)
                try {
                    want = ds::session_tree_words(*session_kwords, static_cast<unsigned long long>(search_batch_) * T::block_words(static_cast<int>(max_children)));
                } catch (const sp::SpError& se) {
                    throw Error(se.code, se.msg);
                }
            }
            if (want > budget || (!session_ && want < per_search + per_search / 4) || want >= (static_cast<uint64_t>(0xFFFFFE) << 2))
                throw Error(CATTUS_B200_ENOMEM, "device search: " + std::to_string(n_slots) + " games x 3 tree buffers of " + std::to_string(want) +
                                                    " words do not fit the device (or its 2^26-word tree address space); lower device_games");
            pool_words_ = static_cast<uint32_t>(want);

            alloc(d_rules_, std::max<size_t>(rules_bytes, 16));
            CB2_CUDA(cudaMemcpy(d_rules_, rules_blob, rules_bytes, cudaMemcpyHostToDevice));
            alloc(d_slots_, sizeof(ds::SlotState) * n_slots);
            CB2_CUDA(cudaMemset(d_slots_, 0, sizeof(ds::SlotState) * n_slots));
            alloc(d_pools_, static_cast<size_t>(n_slots) * 3u * pool_words_ * 4u + 1024u);  // + slack: select fetches a node's first 32 child rows before it knows the count
            const uint32_t path_cap = Rules::kChess ? 256u : max_children + 2u;
            alloc(d_paths_, sizeof(ds::PathStep) * static_cast<size_t>(n_slots) * path_cap);
            alloc(d_noise_, sizeof(float) * static_cast<size_t>(n_slots) * max_children);
            const uint32_t hist_cap = Rules::kChess ? 128u : 1u;
            alloc(d_hist_, sizeof(typename Rules::Pos) * static_cast<size_t>(n_slots) * hist_cap);
            cmd_stride_ = ds::cmd_stride_for(max_children);
            result_stride_ = analysis ? ds::analysis_stride_for(max_children, search_batch_) : ds::result_stride_for(max_children);
            if (search_batch_ > 1) {  // per-descent records and paths, and a virtual count per child row of each slot's tree
                alloc(d_descents_, sizeof(ds::BatchDescent) * static_cast<size_t>(n_slots) * search_batch_);
                alloc(d_bpaths_, sizeof(ds::PathStep) * static_cast<size_t>(n_slots) * search_batch_ * path_cap);
                alloc(d_vcount_, sizeof(uint32_t) * static_cast<size_t>(n_slots) * (pool_words_ >> 2));
                CB2_CUDA(cudaMemset(d_vcount_, 0, sizeof(uint32_t) * static_cast<size_t>(n_slots) * (pool_words_ >> 2)));
            }
            if (roots_cap) {
                roots_cap_ = roots_cap;
                CB2_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&h_roots_), sizeof(typename Rules::Pos) * roots_cap_ * n_bufs_, cudaHostAllocDefault));
            }
            cmd_bytes_ = 16 + static_cast<size_t>(n_slots) * cmd_stride_;
            result_buf_bytes_ = static_cast<size_t>(n_slots) * result_stride_;
            CB2_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&h_results_), result_buf_bytes_ * n_bufs_, cudaHostAllocMapped));
            uint8_t* d_results = nullptr;
            CB2_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&d_results), h_results_, 0));
            CB2_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&h_cmds_), cmd_bytes_ * n_bufs_, cudaHostAllocDefault));
            CB2_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&h_status_), 64 * n_bufs_, cudaHostAllocDefault));
            std::memset(h_status_, 0, 64 * n_bufs_);
            events_.resize(n_bufs_);
            for (auto& ev : events_) CB2_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            // a session's begin runs before the first minibatch of its search, in the same wave
            const uint32_t begin_lead = (session_ || std::getenv("CATTUS_B200_DSEARCH_SERIAL_BEGIN")) ? 0u : 1u;
            if (session_) {
                CB2_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&h_session_), sizeof(ds::SessionCtl) + ds::kSnapshotHdr + result_stride_, cudaHostAllocMapped));
                std::memset(h_session_, 0, sizeof(ds::SessionCtl) + ds::kSnapshotHdr + result_stride_);
                CB2_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&d_session_), h_session_, 0));
            }
            uint32_t visit_budget = 24;  // measured on hex5 (sim_num 1400, whole games): 24 -> 57.1 M sims/s, 48 -> 54.4 M, 96 -> 49.4 M
            if (const char* vb = std::getenv("CATTUS_B200_DSEARCH_VISIT_BUDGET")) visit_budget = static_cast<uint32_t>(std::max(1, std::atoi(vb)));

            for (uint32_t k = 0; k < n_pops_; ++k) {
                DsPopulation<Rules>& P = pop_[k];
                const uint32_t base = k == 0 ? 0 : split_, cnt = k == 0 ? split_ : n_slots - split_;
                ds::Params<Rules>& p = P.p;
                std::memset(&p, 0, sizeof(p));
                CB2_CUDA(cudaStreamCreateWithFlags(&P.stream, cudaStreamNonBlocking));
                alloc(P.d_cmds, cmd_bytes_);
                CB2_CUDA(cudaMemset(P.d_cmds, 0, 16));
                alloc(P.d_status, 64);
                CB2_CUDA(cudaMemset(P.d_status, 0, 64));
                p.rules = d_rules_;
                p.slots = static_cast<ds::SlotState*>(d_slots_) + base;
                p.n_slots = cnt;
                p.slot_base = base;
                p.pools = static_cast<uint32_t*>(d_pools_) + static_cast<size_t>(base) * 3u * pool_words_;
                p.pool_words = pool_words_;
                p.paths = static_cast<ds::PathStep*>(d_paths_) + static_cast<size_t>(base) * path_cap;
                p.path_cap = path_cap;
                p.noise = static_cast<float*>(d_noise_) + static_cast<size_t>(base) * max_children;
                p.max_children = max_children;
                p.hist = static_cast<typename Rules::Pos*>(d_hist_) + static_cast<size_t>(base) * hist_cap;
                p.hist_cap = hist_cap;
                p.n_evals = n_evals_;
                for (uint32_t e = 0; e < 2; ++e) {
                    const Engine::ResidentIo& io = P.io[e < n_evals_ ? e : 0];
                    p.eval[e].n_ptr = reinterpret_cast<uint32_t*>(io.d_block);
                    p.eval[e].recs = io.d_block + 16 + 8;
                    p.eval[e].values = io.d_values;
                    p.eval[e].probs = io.d_probs;
                    p.eval[e].rec_bytes = io.rec_bytes;
                    p.eval[e].prob_stride = io.moves < max_children ? io.moves : max_children;
                    p.eval[e].max_rows = io.max_batch;
                    p.eval[e].plane_words = io.plane_words;
                    p.sim_num[e] = session_ ? 0u : params[e].sim_num;
                    p.explore[e] = params[e].explore_factor;
                    p.noise_eps[e] = params[e].noise_eps;
                    p.cache[e] = ds::CacheIo{};
                }
                // ValueFuncCache in HBM, one per evaluator and population (cfg.cache_size entries over the populations, rounded up
                // to whole buckets): a population's probes (select) and inserts (expand) never overlap, two populations' would
                if (cfg.cache_size) {
                    uint32_t buckets = 1;
                    while (static_cast<uint64_t>(buckets) * ds::kCacheWays * n_pops_ < cfg.cache_size) buckets <<= 1;
                    for (uint32_t e = 0; e < n_evals_; ++e) {
                        ds::CacheIo& c = p.cache[e];
                        c.entry_bytes = (40u + 4u * max_children + 15u) & ~15u;
                        alloc(P.d_cache_meta[e], static_cast<size_t>(buckets) * 32u);
                        CB2_CUDA(cudaMemset(P.d_cache_meta[e], 0, static_cast<size_t>(buckets) * 32u));
                        alloc(P.d_cache_entries[e], static_cast<size_t>(buckets) * ds::kCacheWays * c.entry_bytes);
                        c.meta = static_cast<uint32_t*>(P.d_cache_meta[e]);
                        c.entries = static_cast<uint8_t*>(P.d_cache_entries[e]);
                        c.bucket_mask = buckets - 1;
                        c.enabled = 1;
                    }
                }
                p.cmds = static_cast<const uint8_t*>(P.d_cmds);
                p.cmd_stride = cmd_stride_;
                p.results = d_results;
                p.result_stride = result_stride_;
                p.n_result_bufs = n_bufs_;
                p.result_buf_bytes = result_buf_bytes_;
                p.done_count = static_cast<uint32_t*>(P.d_status);
                p.error = static_cast<uint32_t*>(P.d_status) + 1;
                p.max_used = static_cast<uint32_t*>(P.d_status) + 2;
                p.counters = reinterpret_cast<unsigned long long*>(static_cast<uint8_t*>(P.d_status) + 16);
                // begin (per-move commands: tree reuse copies subtrees) runs on a side branch of the wave graph, beside select /
                // evaluator / expand; its slots take part from the population's next wave on
                p.begin_lead = begin_lead;
                p.visit_budget = visit_budget;
                if (roots_cap_) {
                    alloc(P.d_roots, sizeof(typename Rules::Pos) * roots_cap_);
                    p.roots = static_cast<const typename Rules::Pos*>(P.d_roots);
                }
                if (analysis) {
                    p.analysis = 1;
                    p.pv_max = std::min<uint32_t>(analysis->pv_max, ds::kPvMax);
                }
                if (search_batch_ > 1) {
                    p.search_batch.side[0] = side_batch_[0];
                    p.search_batch.side[1] = side_batch_[1];
                    p.search_batch.max = search_batch_;
                    p.descents = static_cast<ds::BatchDescent*>(d_descents_) + static_cast<size_t>(base) * search_batch_;
                    p.bpaths = static_cast<ds::PathStep*>(d_bpaths_) + static_cast<size_t>(base) * search_batch_ * path_cap;
                    p.vcount = static_cast<uint32_t*>(d_vcount_) + static_cast<size_t>(base) * (pool_words_ >> 2);
                }
                if (session_) {
                    p.session = reinterpret_cast<volatile ds::SessionCtl*>(d_session_);
                    p.snapshot = d_session_ + sizeof(ds::SessionCtl);
                }
                if (begin_lead) {
                    CB2_CUDA(cudaStreamCreateWithFlags(&P.side, cudaStreamNonBlocking));
                    CB2_CUDA(cudaEventCreateWithFlags(&P.fork, cudaEventDisableTiming));
                    CB2_CUDA(cudaEventCreateWithFlags(&P.join, cudaEventDisableTiming));
                }
                capture(P);
            }
            setup_seconds_ = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        } catch (...) {
            destroy();
            throw;
        }
    }
    ~DsCudaBackend() { destroy(); }
    DsCudaBackend(const DsCudaBackend&) = delete;
    DsCudaBackend& operator=(const DsCudaBackend&) = delete;

    uint32_t n_slots() const { return n_slots_; }
    uint32_t max_children() const { return max_children_; }
    uint32_t depth() const { return depth_; }
    uint32_t pool_words() const { return pool_words_; }
    uint32_t populations() const { return n_pops_; }
    uint32_t population_of(uint32_t slot) const { return slot >= split_ ? 1u : 0u; }
    double setup_seconds() const { return setup_seconds_; }
    uint8_t* cmd_block(uint32_t wave) { return h_cmds_ + static_cast<size_t>(wave % n_bufs_) * cmd_bytes_; }
    // root upload: where the host stages a wave's root histories (roots_cap() positions), uploaded by submit()
    typename Rules::Pos* roots_block(uint32_t wave) { return h_roots_ + static_cast<size_t>(wave % n_bufs_) * roots_cap_; }
    uint32_t roots_cap() const { return roots_cap_; }

    void submit(uint32_t wave, uint32_t pop, uint32_t n_cmds, uint32_t n_roots = 0) {
        const uint32_t b = wave % n_bufs_;
        DsPopulation<Rules>& P = pop_[pop];
        wave_pop_[b] = pop;
        if (n_roots)  // the previous wave's begin kernel is done with the buffer: same stream, earlier graph
            CB2_CUDA(cudaMemcpyAsync(P.d_roots, roots_block(wave), sizeof(typename Rules::Pos) * n_roots, cudaMemcpyHostToDevice, P.stream));
        CB2_CUDA(cudaMemcpyAsync(P.d_cmds, cmd_block(wave), 16 + static_cast<size_t>(n_cmds) * cmd_stride_, cudaMemcpyHostToDevice, P.stream));
        CB2_CUDA(cudaGraphLaunch(P.graph, P.stream));
        CB2_CUDA(cudaMemcpyAsync(h_status_ + 64 * b, P.d_status, 64, cudaMemcpyDeviceToHost, P.stream));
        CB2_CUDA(cudaEventRecord(events_[b], P.stream));
        waves_ += 1;
    }
    const uint8_t* wait(uint32_t wave, uint32_t* n_done) {
        const uint32_t b = wave % n_bufs_;
        const cudaError_t e = cudaEventSynchronize(events_[b]);
        if (e != cudaSuccess) throw Error(CATTUS_B200_ECUDA, std::string("device search wave failed: ") + cudaGetErrorString(e));
        const uint32_t* st = reinterpret_cast<const uint32_t*>(h_status_ + 64 * b);
        if (st[1]) {
            std::string what;
            if (st[1] & ds::kErrPool) what += " tree pool exhausted (raise device_tree_kwords or lower device_games);";
            if (st[1] & ds::kErrPath) what += " search path deeper than the path buffer;";
            if (st[1] & ds::kErrRows) what += " evaluator batch overflow;";
            if (st[1] & ds::kErrNoise) what += " noise sample size does not match the root;";
            throw Error(CATTUS_B200_ERANGE, "device search:" + what);
        }
        *n_done = st[0];
        return h_results_ + static_cast<size_t>(b) * result_buf_bytes_;
    }
    void read_counters(unsigned long long out[4]) {
        for (int i = 0; i < 4; ++i) out[i] = 0;
        for (uint32_t k = 0; k < n_pops_; ++k) {
            unsigned long long c[4];
            uint32_t hw = 0;
            CB2_CUDA(cudaStreamSynchronize(pop_[k].stream));
            CB2_CUDA(cudaMemcpy(c, static_cast<uint8_t*>(pop_[k].d_status) + 16, sizeof(c), cudaMemcpyDeviceToHost));
            CB2_CUDA(cudaMemcpy(&hw, static_cast<uint8_t*>(pop_[k].d_status) + 8, sizeof(hw), cudaMemcpyDeviceToHost));
            for (int i = 0; i < 4; ++i) out[i] += c[i];
            max_used_ = std::max(max_used_, hw);
        }
    }
    uint32_t max_used() const { return max_used_; }
    uint64_t waves() const { return waves_; }
    uint32_t kernels_per_wave() const { return kernels_per_wave_; }
    // a session's control words and snapshot (mapped pinned memory the device reads and writes while the host does)
    volatile ds::SessionCtl* session_ctl() { return reinterpret_cast<volatile ds::SessionCtl*>(h_session_); }
    const uint8_t* snapshot() const { return h_session_ + sizeof(ds::SessionCtl); }
    void bind_thread() { CB2_CUDA(cudaSetDevice(device_)); }
    // A session goes on after a search that met a device error (ErrBits): the sticky error word is cleared, and so are the
    // virtual counts the failed minibatch left behind (its backup never ran).  The next search starts from a fresh root.
    void clear_error() {
        DsPopulation<Rules>& P = pop_[0];
        CB2_CUDA(cudaMemsetAsync(static_cast<uint32_t*>(P.d_status) + 1, 0, 4, P.stream));
        if (d_vcount_) CB2_CUDA(cudaMemsetAsync(d_vcount_, 0, sizeof(uint32_t) * static_cast<size_t>(n_slots_) * (pool_words_ >> 2), P.stream));
        CB2_CUDA(cudaStreamSynchronize(P.stream));
    }
    int error_code(const std::exception& e) const {
        const Error* ce = dynamic_cast<const Error*>(&e);
        return ce ? ce->code : CATTUS_B200_EDEVICE;
    }

  private:
    void alloc(void*& ptr, size_t bytes) {
        const cudaError_t e = cudaMalloc(&ptr, bytes);
        if (e != cudaSuccess) {
            ptr = nullptr;
            throw Error(CATTUS_B200_ENOMEM, "device search: cudaMalloc(" + std::to_string(bytes) + "): " + cudaGetErrorString(e));
        }
    }
    void capture(DsPopulation<Rules>& P) {
        const uint32_t blocks = (P.p.n_slots + 3u) / 4u;
        cudaGraph_t g = nullptr;
        CB2_CUDA(cudaStreamBeginCapture(P.stream, cudaStreamCaptureModeThreadLocal));
        try {
            for (uint32_t e = 0; e < n_evals_; ++e) CB2_CUDA(cudaMemsetAsync(P.io[e].d_block, 0, 4, P.stream));
            CB2_CUDA(cudaMemsetAsync(P.d_status, 0, 4, P.stream));
            if (P.p.begin_lead) {
                CB2_CUDA(cudaEventRecord(P.fork, P.stream));
                CB2_CUDA(cudaStreamWaitEvent(P.side, P.fork, 0));
                ds_begin_kernel<Rules><<<blocks, 128, 0, P.side>>>(P.p);
                CB2_CUDA(cudaEventRecord(P.join, P.side));
            } else if (session_) {
                ds_begin_session_kernel<Rules><<<blocks, 128, 0, P.stream>>>(P.p);
            } else {
                ds_begin_kernel<Rules><<<blocks, 128, 0, P.stream>>>(P.p);
            }
            if (search_batch_ > 1)
                ds_select_batch_kernel<Rules><<<blocks, 128, 0, P.stream>>>(P.p);
            else
                ds_select_kernel<Rules><<<blocks, 128, 0, P.stream>>>(P.p);
            for (uint32_t e = 0; e < n_evals_; ++e) eng_[e]->resident_enqueue(P.io[e].lane, P.stream);
            if (search_batch_ > 1)
                ds_expand_batch_kernel<Rules><<<blocks, 128, 0, P.stream>>>(P.p);
            else
                ds_expand_kernel<Rules><<<blocks, 128, 0, P.stream>>>(P.p);
            if (P.p.begin_lead) CB2_CUDA(cudaStreamWaitEvent(P.stream, P.join, 0));
            CB2_CUDA(cudaGetLastError());
        } catch (...) {
            cudaStreamEndCapture(P.stream, &g);
            if (g) cudaGraphDestroy(g);
            throw;
        }
        cudaError_t ce = cudaStreamEndCapture(P.stream, &g);
        if (ce != cudaSuccess) throw Error(CATTUS_B200_ECUDA, std::string("device search: graph capture failed: ") + cudaGetErrorString(ce));
        ce = cudaGraphInstantiate(&P.graph, g, 0);
        cudaGraphDestroy(g);
        if (ce != cudaSuccess) throw Error(CATTUS_B200_ECUDA, std::string("device search: graph instantiate failed: ") + cudaGetErrorString(ce));
        kernels_per_wave_ = 3;
        for (uint32_t e = 0; e < n_evals_; ++e) kernels_per_wave_ += P.io[e].kernels;
    }
    void destroy() {
        for (DsPopulation<Rules>& P : pop_) {
            if (P.stream) cudaStreamSynchronize(P.stream);
            if (P.graph) cudaGraphExecDestroy(P.graph);
            P.graph = nullptr;
            if (P.stream) cudaStreamDestroy(P.stream);
            if (P.side) cudaStreamDestroy(P.side);
            P.stream = P.side = nullptr;
            if (P.fork) cudaEventDestroy(P.fork);
            if (P.join) cudaEventDestroy(P.join);
            P.fork = P.join = nullptr;
            for (void** q : {&P.d_cmds, &P.d_status, &P.d_cache_meta[0], &P.d_cache_meta[1], &P.d_cache_entries[0], &P.d_cache_entries[1], &P.d_roots}) {
                if (*q) cudaFree(*q);
                *q = nullptr;
            }
            for (uint32_t e = 0; e < 2; ++e)
                if (P.io[e].lane >= 0 && eng_[e]) {
                    eng_[e]->resident_release(P.io[e].lane);
                    P.io[e].lane = -1;
                }
        }
        for (auto& ev : events_)
            if (ev) cudaEventDestroy(ev);
        events_.clear();
        for (void** q : {&d_rules_, &d_slots_, &d_pools_, &d_paths_, &d_noise_, &d_hist_, &d_descents_, &d_bpaths_, &d_vcount_}) {
            if (*q) cudaFree(*q);
            *q = nullptr;
        }
        if (h_results_) cudaFreeHost(h_results_);
        if (h_cmds_) cudaFreeHost(h_cmds_);
        if (h_status_) cudaFreeHost(h_status_);
        if (h_roots_) cudaFreeHost(h_roots_);
        if (h_session_) cudaFreeHost(h_session_);
        h_results_ = h_cmds_ = h_status_ = h_session_ = d_session_ = nullptr;
        h_roots_ = nullptr;
    }

    DsPopulation<Rules> pop_[2];
    Engine* eng_[2] = {nullptr, nullptr};
    uint32_t n_evals_ = 1, n_pops_ = 1, split_ = 0, depth_ = 2, n_bufs_ = 3, max_children_ = 0, n_slots_ = 0, pool_words_ = 0, cmd_stride_ = 0,
             result_stride_ = 0, kernels_per_wave_ = 0, roots_cap_ = 0, search_batch_ = 1;
    uint32_t side_batch_[2] = {1, 1};  // search_batch_ is the larger
    size_t cmd_bytes_ = 0, result_buf_bytes_ = 0;
    void *d_rules_ = nullptr, *d_slots_ = nullptr, *d_pools_ = nullptr, *d_paths_ = nullptr, *d_noise_ = nullptr, *d_hist_ = nullptr;
    void *d_descents_ = nullptr, *d_bpaths_ = nullptr, *d_vcount_ = nullptr;
    uint8_t *h_results_ = nullptr, *h_cmds_ = nullptr, *h_status_ = nullptr, *h_session_ = nullptr, *d_session_ = nullptr;
    int device_ = 0;
    bool session_ = false;
    typename Rules::Pos* h_roots_ = nullptr;
    std::vector<cudaEvent_t> events_;
    std::vector<uint32_t> wave_pop_;
    uint64_t waves_ = 0;
    uint32_t max_used_ = 0;
    double setup_seconds_ = 0.0;
};

template <class Rules>
static void dsearch_run_rules(const Rules& rules, const void* blob, size_t blob_bytes, uint32_t max_children, Engine* e1, Engine* e2,
                              const cattus_b200_selfplay_cfg& cfg, const sp::Params params[2], const uint32_t search_batch[2], sp::Shared& sh) {
    const uint32_t stride = std::max<uint32_t>(1, cfg.game_stride);
    const uint32_t my_games = cfg.games_num > cfg.first_game ? (cfg.games_num - cfg.first_game + stride - 1) / stride : 0;
    if (my_games == 0) return;
    uint32_t max_batch = 0xFFFFFFFFu;
    for (Engine* e : {e1, e2}) {
        if (!e) continue;
        cattus_b200_info info;
        e->get_info(&info);
        max_batch = std::min(max_batch, info.max_batch);
    }
    const uint32_t n_slots = ds::selfplay_slots(cfg.device_games, my_games, max_batch, std::max(search_batch[0], search_batch[1]));
    const auto t0 = std::chrono::steady_clock::now();
    DsCudaBackend<Rules> be(blob, blob_bytes, max_children, e1, e2, cfg, params, n_slots, 0, search_batch);
    if (std::getenv("CATTUS_B200_DSEARCH_PROFILE"))
        std::fprintf(stderr, "device search: %u slots in %u population(s), %u words per tree buffer, set up in %.3f s\n", n_slots, be.populations(),
                     be.pool_words(), be.setup_seconds());
    ds::Driver<Rules, DsCudaBackend<Rules>> drv(rules, cfg, params, be, sh, nullptr, search_batch);
    drv.run();
    const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    const uint64_t waves = be.waves();
    if (std::getenv("CATTUS_B200_DSEARCH_PROFILE"))
        std::fprintf(stderr, "device search: fullest tree buffer used %u of %u words (%.0f %%)\n", be.max_used(), be.pool_words(),
                     100.0 * be.max_used() / std::max(1u, be.pool_words()));
    e1->note_resident(waves, sh.evaluations, waves * be.kernels_per_wave(), waves ? secs / static_cast<double>(waves) : 0.0);
}

// Batched analysis of given positions (dsearch_analysis.hpp) on model's device: the self-play backend with the analysis
// result layout and kCmdSetRoot's root upload.
template <class Rules>
static void analyse_rules(const Rules& rules, const void* blob, size_t blob_bytes, uint32_t max_children, Engine* e, const cattus_b200_selfplay_cfg& cfg,
                          uint32_t search_batch, uint32_t n, const char* const* fens, const uint16_t* moves, const uint32_t* move_offsets, std::vector<ds::AnalysisResult>& out) {
    const sp::Params params[2] = {ds::analysis_params(cfg), ds::analysis_params(cfg)};
    const auto hist = ds::analysis_histories(rules, n, fens, moves, move_offsets);
    cattus_b200_info info;
    e->get_info(&info);
    if (info.game != cfg.game || (cfg.game == CATTUS_B200_GAME_HEX && info.board_size != cfg.board_size))
        throw Error(CATTUS_B200_EINVAL, "analysis: the model was made for another game or board size than cfg");
    const uint32_t n_slots = ds::analysis_slots(cfg.device_games, n, info.max_batch, search_batch);
    if (n == 0) {
        out.clear();
        return;
    }
    // a wave's root upload: a few history positions per slot on average; a longer run of long histories waits a wave
    const ds::AnalysisOpts opts{ds::kPvMax};
    const uint32_t sides[2] = {search_batch, search_batch};
    const auto t0 = std::chrono::steady_clock::now();
    DsCudaBackend<Rules> be(blob, blob_bytes, max_children, e, nullptr, cfg, params, n_slots, n_slots * 8u + ds::hist_cap_for<Rules>(), sides, &opts);
    ds::AnalysisDriver<Rules, DsCudaBackend<Rules>> drv(rules, params[0], be, hist, out, search_batch);
    drv.run();
    const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    const uint64_t waves = be.waves();
    e->note_resident(waves, drv.counters()[1], waves * be.kernels_per_wave(), waves ? secs / static_cast<double>(waves) : 0.0);
}

void analyse_run(cattus_b200_t* m, const cattus_b200_selfplay_cfg& cfg, uint32_t search_batch, uint32_t n, const char* const* fens, const uint16_t* moves,
                 const uint32_t* move_offsets, std::vector<ds::AnalysisResult>& out) {
    try {
        if (!m) throw Error(CATTUS_B200_EINVAL, "null evaluator handle (there is no CPU fallback)");
        if (cfg.struct_size != sizeof(cattus_b200_selfplay_cfg)) throw Error(CATTUS_B200_EINVAL, "selfplay cfg struct_size mismatch");
        if (cfg.game == CATTUS_B200_GAME_HEX) {
            const int s = static_cast<int>(cfg.board_size);
            if (s < 2 || s > 11) throw Error(CATTUS_B200_EINVAL, "hex board_size must be 2..11");
            if (s <= 8) {
                sp::HexRulesT<uint64_t> rules(s);
                analyse_rules(rules, &rules, sizeof(rules), static_cast<uint32_t>(s * s), m->engine, cfg, search_batch, n, fens, moves, move_offsets, out);
            } else {
                sp::HexRulesT<sp::u128> rules(s);
                analyse_rules(rules, &rules, sizeof(rules), static_cast<uint32_t>(s * s), m->engine, cfg, search_batch, n, fens, moves, move_offsets, out);
            }
        } else if (cfg.game == CATTUS_B200_GAME_CHESS) {
            sp::ChessRules rules;
            analyse_rules(rules, &sp::chess_tables(), sizeof(sp::ChessTables), static_cast<uint32_t>(sp::ChessRules::kMaxMoves), m->engine, cfg, search_batch,
                          n, fens, moves, move_offsets, out);
        } else if (cfg.game == CATTUS_B200_GAME_TTT) {
            sp::TttRules rules;
            analyse_rules(rules, &rules, sizeof(rules), 9u, m->engine, cfg, search_batch, n, fens, moves, move_offsets, out);
        } else {
            throw Error(CATTUS_B200_EINVAL, "unknown game");
        }
    } catch (const sp::SpError& e) {
        throw Error(e.code ? e.code : CATTUS_B200_EINVAL, e.msg);
    }
}

// A match from openings (dsearch_match.hpp) between e1 (A) and e2 (B; nullptr: the same handle): the self-play backend
// and result layout with kCmdSetRoot's root upload.
template <class Rules>
static void match_rules(const Rules& rules, const void* blob, size_t blob_bytes, uint32_t max_children, Engine* e1, Engine* e2,
                        const cattus_b200_selfplay_cfg& cfg, const cattus_b200_match_side* side_b, const uint32_t search_batch[2], uint32_t n,
                        const char* const* fens, const uint16_t* moves, const uint32_t* move_offsets, ds::MatchResult& out) {
    const auto t0 = std::chrono::steady_clock::now();
    sp::Params params[2];
    ds::match_params(cfg, side_b, params);
    uint32_t max_batch = 0xFFFFFFFFu;
    for (Engine* e : {e1, e2}) {
        if (!e) continue;
        cattus_b200_info info;
        e->get_info(&info);
        if (info.game != cfg.game || (cfg.game == CATTUS_B200_GAME_HEX && info.board_size != cfg.board_size))
            throw Error(CATTUS_B200_EINVAL, "match: a model was made for another game or board size than cfg");
        if (cfg.device_games > info.max_batch)
            throw Error(CATTUS_B200_ERANGE, "device search: device_games (" + std::to_string(cfg.device_games) + ") exceeds the evaluator's max_batch (" +
                                                std::to_string(info.max_batch) + ")");
        max_batch = std::min(max_batch, info.max_batch);
    }
    if (e2 && e2->device() != e1->device()) throw Error(CATTUS_B200_EINVAL, "match: both models must live on the same device");
    const auto openings = ds::match_openings(rules, n, fens, moves, move_offsets, out.opening_status);
    const uint32_t games = ds::match_games(out.opening_status);
    if (games) {
        const uint32_t n_slots = ds::analysis_slots(cfg.device_games, games, max_batch, std::max(search_batch[0], search_batch[1]));
        // a wave's root upload: a few history positions per slot on average; a longer run of long histories waits a wave
        DsCudaBackend<Rules> be(blob, blob_bytes, max_children, e1, e2, cfg, params, n_slots, n_slots * 8u + ds::hist_cap_for<Rules>(), search_batch);
        ds::match_play(rules, cfg, params, be, openings, out, search_batch);
        const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        const uint64_t waves = be.waves();
        e1->note_resident(waves, out.evaluations, waves * be.kernels_per_wave(), waves ? secs / static_cast<double>(waves) : 0.0);
    }
    out.seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}

void match_run(cattus_b200_t* ma, cattus_b200_t* mb, const cattus_b200_selfplay_cfg& cfg, const cattus_b200_match_side* side_b,
               const uint32_t search_batch[2], uint32_t n, const char* const* fens, const uint16_t* moves, const uint32_t* move_offsets,
               ds::MatchResult& out) {
    try {
        if (!ma) throw Error(CATTUS_B200_EINVAL, "null evaluator handle (there is no CPU fallback)");
        if (cfg.struct_size != sizeof(cattus_b200_selfplay_cfg)) throw Error(CATTUS_B200_EINVAL, "selfplay cfg struct_size mismatch");
        Engine* e1 = ma->engine;
        Engine* e2 = (mb && mb != ma) ? mb->engine : nullptr;
        if (cfg.game == CATTUS_B200_GAME_HEX) {
            const int s = static_cast<int>(cfg.board_size);
            if (s < 2 || s > 11) throw Error(CATTUS_B200_EINVAL, "hex board_size must be 2..11");
            if (s <= 8) {
                sp::HexRulesT<uint64_t> rules(s);
                match_rules(rules, &rules, sizeof(rules), static_cast<uint32_t>(s * s), e1, e2, cfg, side_b, search_batch, n, fens, moves, move_offsets, out);
            } else {
                sp::HexRulesT<sp::u128> rules(s);
                match_rules(rules, &rules, sizeof(rules), static_cast<uint32_t>(s * s), e1, e2, cfg, side_b, search_batch, n, fens, moves, move_offsets, out);
            }
        } else if (cfg.game == CATTUS_B200_GAME_CHESS) {
            sp::ChessRules rules;
            match_rules(rules, &sp::chess_tables(), sizeof(sp::ChessTables), static_cast<uint32_t>(sp::ChessRules::kMaxMoves), e1, e2, cfg, side_b,
                        search_batch, n, fens, moves, move_offsets, out);
        } else if (cfg.game == CATTUS_B200_GAME_TTT) {
            sp::TttRules rules;
            match_rules(rules, &rules, sizeof(rules), 9u, e1, e2, cfg, side_b, search_batch, n, fens, moves, move_offsets, out);
        } else {
            throw Error(CATTUS_B200_EINVAL, "unknown game");
        }
    } catch (const sp::SpError& e) {
        throw Error(e.code ? e.code : CATTUS_B200_EINVAL, e.msg);
    }
}

// A session (dsearch_session.hpp) on model's device: the analysis backend with one slot, the session's begin and the
// session's tree size; the driver owns the backend and its evaluator lane.
template <class Rules>
static std::unique_ptr<ds::SessionBase> session_rules(const Rules& rules, const void* blob, size_t blob_bytes, uint32_t max_children, Engine* e,
                                                      const cattus_b200_selfplay_cfg& cfg, const cattus_b200_session_opts* opts) {
    cattus_b200_selfplay_cfg c = cfg;
    c.sim_num = std::max<uint32_t>(c.sim_num, 2u);  // not used by a session; analysis_params checks it
    const sp::Params params[2] = {ds::analysis_params(c), ds::analysis_params(c)};
    cattus_b200_info info;
    e->get_info(&info);
    if (info.game != cfg.game || (cfg.game == CATTUS_B200_GAME_HEX && info.board_size != cfg.board_size))
        throw Error(CATTUS_B200_EINVAL, "session: the model was made for another game or board size than cfg");
    if (info.n_streams < 2)
        throw Error(CATTUS_B200_EINVAL, "session: a session holds one evaluator lane for its lifetime; create the model with n_streams >= 2");
    const uint32_t L = ds::session_search_batch(opts, info.max_batch);
    const uint32_t sides[2] = {L, L};
    const ds::AnalysisOpts aopts{ds::kPvMax};
    const uint32_t kwords = opts->tree_kwords;
    std::unique_ptr<DsCudaBackend<Rules>> be(
        new DsCudaBackend<Rules>(blob, blob_bytes, max_children, e, nullptr, c, params, 1, ds::hist_cap_for<Rules>(), sides, &aopts, &kwords));
    return std::unique_ptr<ds::SessionBase>(new ds::SessionDriver<Rules, DsCudaBackend<Rules>>(rules, params[0], std::move(be), L));
}

std::unique_ptr<ds::SessionBase> session_create(cattus_b200_t* m, const cattus_b200_selfplay_cfg& cfg, const cattus_b200_session_opts* opts) {
    try {
        if (!m) throw Error(CATTUS_B200_EINVAL, "null evaluator handle (there is no CPU fallback)");
        if (cfg.struct_size != sizeof(cattus_b200_selfplay_cfg)) throw Error(CATTUS_B200_EINVAL, "selfplay cfg struct_size mismatch");
        if (cfg.game == CATTUS_B200_GAME_HEX) {
            const int s = static_cast<int>(cfg.board_size);
            if (s < 2 || s > 11) throw Error(CATTUS_B200_EINVAL, "hex board_size must be 2..11");
            if (s <= 8) {
                sp::HexRulesT<uint64_t> rules(s);
                return session_rules(rules, &rules, sizeof(rules), static_cast<uint32_t>(s * s), m->engine, cfg, opts);
            }
            sp::HexRulesT<sp::u128> rules(s);
            return session_rules(rules, &rules, sizeof(rules), static_cast<uint32_t>(s * s), m->engine, cfg, opts);
        } else if (cfg.game == CATTUS_B200_GAME_CHESS) {
            sp::ChessRules rules;
            return session_rules(rules, &sp::chess_tables(), sizeof(sp::ChessTables), static_cast<uint32_t>(sp::ChessRules::kMaxMoves), m->engine, cfg, opts);
        } else if (cfg.game == CATTUS_B200_GAME_TTT) {
            sp::TttRules rules;
            return session_rules(rules, &rules, sizeof(rules), 9u, m->engine, cfg, opts);
        }
        throw Error(CATTUS_B200_EINVAL, "unknown game");
    } catch (const sp::SpError& e) {
        throw Error(e.code ? e.code : CATTUS_B200_EINVAL, e.msg);
    }
}

void dsearch_run(cattus_b200_t* m1, cattus_b200_t* m2, const cattus_b200_selfplay_cfg& cfg, const sp::Params params[2], const uint32_t search_batch[2],
                 sp::Shared& sh) {
    try {
        if (!m1) throw Error(CATTUS_B200_EINVAL, "null evaluator handle (there is no CPU fallback)");
        Engine* e1 = m1->engine;
        Engine* e2 = (m2 && m2 != m1) ? m2->engine : nullptr;
        if (cfg.game == CATTUS_B200_GAME_HEX) {
            const int s = static_cast<int>(cfg.board_size);
            if (s <= 8) {
                sp::HexRulesT<uint64_t> rules(s);
                dsearch_run_rules(rules, &rules, sizeof(rules), static_cast<uint32_t>(s * s), e1, e2, cfg, params, search_batch, sh);
            } else {
                sp::HexRulesT<sp::u128> rules(s);
                dsearch_run_rules(rules, &rules, sizeof(rules), static_cast<uint32_t>(s * s), e1, e2, cfg, params, search_batch, sh);
            }
        } else if (cfg.game == CATTUS_B200_GAME_CHESS) {
            sp::ChessRules rules;
            dsearch_run_rules(rules, &sp::chess_tables(), sizeof(sp::ChessTables), static_cast<uint32_t>(sp::ChessRules::kMaxMoves), e1, e2, cfg, params, search_batch, sh);
        } else {
            sp::TttRules rules;
            dsearch_run_rules(rules, &rules, sizeof(rules), 9u, e1, e2, cfg, params, search_batch, sh);
        }
    } catch (const Error& e) {
        throw sp::SpError{e.code, e.what()};
    }
}

}  // namespace cb2
