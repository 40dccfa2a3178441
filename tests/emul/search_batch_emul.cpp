// TEST INFRASTRUCTURE -- never part of the product library.
//
// The batched analysis with minibatches under virtual loss (dsearch_core.hpp's batch_select_slot / batch_expand_slot,
// DESIGN.md section 15) over the host emulation of the device-resident search: analysis_emul.cpp's backend with an
// evaluator batch of n_slots x search_batch rows, the per-descent buffers and the virtual counts.  search_batch 1 runs
// analysis_emul.cpp's backend unchanged.  The CPU tests compare it with tests/batch_oracle.py.
#include "analysis_emul.cpp"

namespace {

template <class Rules>
struct EmulBatchBackend : EmulAnalysisBackend<Rules> {
    using Base = EmulAnalysisBackend<Rules>;
    uint32_t L;
    std::vector<ds::BatchDescent> descents;
    std::vector<ds::PathStep> bpaths;
    std::vector<uint32_t> vcount;

    EmulBatchBackend(const Rules& rules, const void* blob, uint32_t n_slots, uint32_t pool_words, uint32_t depth, const sp::Params params[2],
                     cattus_b200_eval_fn f, uint32_t cache_size, uint32_t roots_cap, uint32_t search_batch)
        : Base(rules, blob, n_slots, pool_words, depth, params, f, nullptr, cache_size, roots_cap), L(search_batch) {
        if (this->n_pops != 1) throw sp::SpError{CATTUS_B200_EINVAL, "emul: minibatches run one population"};
        if (L <= 1) return;
        ds::Params<Rules>& p = this->p;
        const uint32_t rows = n_slots * L;
        for (int e = 0; e < 2; ++e) {
            this->block[e].assign(16 + static_cast<size_t>(rows) * p.eval[e].rec_bytes, 0);
            this->values[e].assign(rows, 0.0f);
            this->probs[e].assign(static_cast<size_t>(rows) * p.max_children, 0.0f);
            p.eval[e].n_ptr = reinterpret_cast<uint32_t*>(this->block[e].data());
            p.eval[e].recs = this->block[e].data() + 16 + 8;
            p.eval[e].values = this->values[e].data();
            p.eval[e].probs = this->probs[e].data();
            p.eval[e].max_rows = rows;
        }
        const uint32_t stride = ds::analysis_stride_for(p.max_children, L);
        this->results.assign(static_cast<size_t>(this->n_bufs) * n_slots * stride, 0);
        p.result_stride = stride;
        p.result_buf_bytes = static_cast<unsigned long long>(n_slots) * stride;
        p.results = this->results.data();
        descents.assign(static_cast<size_t>(n_slots) * L, ds::BatchDescent{});
        bpaths.resize(static_cast<size_t>(n_slots) * L * p.path_cap);
        vcount.assign(static_cast<size_t>(n_slots) * (pool_words >> 2), 0u);
        p.search_batch = L;
        p.descents = descents.data();
        p.bpaths = bpaths.data();
        p.vcount = vcount.data();
    }

    void submit(uint32_t wave, uint32_t pop, uint32_t n_cmds, uint32_t n_roots) {
        if (L <= 1) {
            Base::submit(wave, pop, n_cmds, n_roots);
            return;
        }
        ds::Params<Rules>& p = this->p;
        this->done_count = 0;
        *p.eval[0].n_ptr = 0;
        *p.eval[1].n_ptr = 0;
        decltype(auto) rules = ds::RulesRef<Rules>::get(p.rules);
        if (!p.begin_lead)
            for (uint32_t ci = 0; ci < n_cmds; ++ci) ds::Core<Rules>::begin_slot(rules, p, ci, wave);
        for (uint32_t si = 0; si < p.n_slots; ++si) ds::Core<Rules>::batch_select_slot(rules, p, si, wave);
        if (p.begin_lead)
            for (uint32_t ci = 0; ci < n_cmds; ++ci) ds::Core<Rules>::begin_slot(rules, p, ci, wave);
        this->run_eval(p, this->probs, this->values, 0);
        for (uint32_t si = 0; si < p.n_slots; ++si) ds::Core<Rules>::batch_expand_slot(rules, p, si, wave);
        this->done_per_buf[wave % this->n_bufs] = this->done_count;
    }
};

template <class Rules>
void batch_emul(const Rules& rules, const void* blob, const cattus_b200_selfplay_cfg* cfg, uint32_t search_batch, uint32_t max_batch, uint32_t n,
                const char* const* fens, const uint16_t* moves, const uint32_t* offsets, uint32_t pool_words, uint32_t depth, uint32_t roots_cap,
                cattus_b200_eval_fn f, std::vector<ds::AnalysisResult>& out) {
    const sp::Params params[2] = {ds::analysis_params(*cfg), ds::analysis_params(*cfg)};
    const auto hist = ds::analysis_histories(rules, n, fens, moves, offsets);
    const uint32_t n_slots = ds::analysis_slots(cfg->device_games, n, max_batch, search_batch);
    EmulBatchBackend<Rules> be(rules, blob, n_slots, pool_words, depth, params, f, cfg->cache_size, std::max(roots_cap, ds::hist_cap_for<Rules>()),
                               search_batch);
    ds::AnalysisDriver<Rules, EmulBatchBackend<Rules>> drv(rules, params[0], be, hist, out, search_batch);
    drv.run();
}

}  // namespace

extern "C" {

// opts: the C ABI's options (NULL: one leaf in flight); max_batch: the evaluator batch the slots are checked against
// (cfg->device_games 0 takes max_batch / search_batch of them); depth / roots_cap: analysis_emul_run's knobs
void* search_batch_emul_run(cattus_b200_eval_fn f, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_analysis_opts* opts, uint32_t max_batch,
                            uint32_t n, const char* const* fens, const uint16_t* moves, const uint32_t* offsets, uint32_t pool_words, uint32_t depth,
                            uint32_t roots_cap, int* code) {
    std::unique_ptr<AnalysisEmulResult> r(new AnalysisEmulResult());
    *code = 0;
    try {
        const uint32_t L = ds::analysis_search_batch(opts);
        if (cfg->game == CATTUS_B200_GAME_HEX) {
            if (cfg->board_size <= 8) {
                sp::HexRulesT<uint64_t> rules(static_cast<int>(cfg->board_size));
                batch_emul(rules, &rules, cfg, L, max_batch, n, fens, moves, offsets, pool_words, depth, roots_cap, f, r->res);
            } else {
                sp::HexRulesT<sp::u128> rules(static_cast<int>(cfg->board_size));
                batch_emul(rules, &rules, cfg, L, max_batch, n, fens, moves, offsets, pool_words, depth, roots_cap, f, r->res);
            }
        } else if (cfg->game == CATTUS_B200_GAME_CHESS) {
            sp::ChessRules rules;
            batch_emul(rules, &sp::chess_tables(), cfg, L, max_batch, n, fens, moves, offsets, pool_words, depth, roots_cap, f, r->res);
        } else {
            sp::TttRules rules;
            batch_emul(rules, &rules, cfg, L, max_batch, n, fens, moves, offsets, pool_words, depth, roots_cap, f, r->res);
        }
    } catch (const sp::SpError& e) {
        r->error = e.msg.empty() ? "error" : e.msg;
        *code = e.code;
    }
    return r.release();
}
int search_batch_emul_batches(const void* h, uint32_t k, uint32_t* minibatches, uint32_t* collisions) {
    return ds::analysis_batches(static_cast<const AnalysisEmulResult*>(h)->res, k, minibatches, collisions);
}
}
