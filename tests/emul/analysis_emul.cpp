// TEST INFRASTRUCTURE -- never part of the product library.
//
// The batched analysis (cattus_b200/csrc/dsearch_analysis.hpp) over the host emulation of the device-resident search
// (dsearch_emul.cpp, included whole: its EmulBackend gains the analysis result layout and the root upload here), with a
// callback evaluator.  The CPU tests compare it with oracle/mcts.py's MctsPlayer position by position.
#include "dsearch_emul.cpp"

#include "../../cattus_b200/csrc/dsearch_analysis.hpp"

namespace {

template <class Rules>
struct EmulAnalysisBackend : EmulBackend<Rules> {
    using Base = EmulBackend<Rules>;
    using Pos = typename Rules::Pos;
    std::vector<Pos> roots;
    uint32_t cap;

    EmulAnalysisBackend(const Rules& rules, const void* blob, uint32_t n_slots, uint32_t pool_words, uint32_t depth, const sp::Params params[2],
                        cattus_b200_eval_fn f, void* c, uint32_t cache_size, uint32_t roots_cap)
        : Base(rules, blob, n_slots, pool_words, depth, params, f, c, nullptr, nullptr, cache_size), cap(roots_cap) {
        roots.assign(roots_cap, Pos());
        const uint32_t stride = ds::analysis_stride_for(this->p.max_children);
        this->results.assign(static_cast<size_t>(this->n_bufs) * n_slots * stride, 0);
        for (ds::Params<Rules>* q : {&this->p, &this->p2}) {
            q->result_stride = stride;
            q->result_buf_bytes = static_cast<unsigned long long>(n_slots) * stride;
            q->results = this->results.data();
            q->roots = roots.data();
            q->analysis = 1;
            q->pv_max = ds::kPvMax;
        }
    }
    Pos* roots_block(uint32_t) { return roots.data(); }
    uint32_t roots_cap() const { return cap; }
    void submit(uint32_t wave, uint32_t pop, uint32_t n_cmds, uint32_t) { Base::submit(wave, pop, n_cmds); }
};

struct AnalysisEmulResult {
    std::vector<ds::AnalysisResult> res;
    std::string error;
};

template <class Rules>
void analyse_emul(const Rules& rules, const void* blob, const cattus_b200_selfplay_cfg* cfg, uint32_t n, const char* const* fens, const uint16_t* moves,
                  const uint32_t* offsets, uint32_t n_slots, uint32_t pool_words, uint32_t depth, uint32_t roots_cap, cattus_b200_eval_fn f, void* c,
                  std::vector<ds::AnalysisResult>& out) {
    const sp::Params params[2] = {ds::analysis_params(*cfg), ds::analysis_params(*cfg)};
    const auto hist = ds::analysis_histories(rules, n, fens, moves, offsets);
    EmulAnalysisBackend<Rules> be(rules, blob, n_slots, pool_words, depth, params, f, c, cfg->cache_size,
                                  std::max(roots_cap, ds::hist_cap_for<Rules>()));
    ds::AnalysisDriver<Rules, EmulAnalysisBackend<Rules>> drv(rules, params[0], be, hist, out);
    drv.run();
}

}  // namespace

extern "C" {

// depth: the test knobs of dsearch_emul_run; roots_cap: history positions one wave can upload (raised to the ring size)
void* analysis_emul_run(cattus_b200_eval_fn f, const cattus_b200_selfplay_cfg* cfg, uint32_t n, const char* const* fens, const uint16_t* moves,
                        const uint32_t* offsets, uint32_t n_slots, uint32_t pool_words, uint32_t depth, uint32_t roots_cap) {
    std::unique_ptr<AnalysisEmulResult> r(new AnalysisEmulResult());
    try {
        if (cfg->game == CATTUS_B200_GAME_HEX) {
            if (cfg->board_size <= 8) {
                sp::HexRulesT<uint64_t> rules(static_cast<int>(cfg->board_size));
                analyse_emul(rules, &rules, cfg, n, fens, moves, offsets, n_slots, pool_words, depth, roots_cap, f, nullptr, r->res);
            } else {
                sp::HexRulesT<sp::u128> rules(static_cast<int>(cfg->board_size));
                analyse_emul(rules, &rules, cfg, n, fens, moves, offsets, n_slots, pool_words, depth, roots_cap, f, nullptr, r->res);
            }
        } else if (cfg->game == CATTUS_B200_GAME_CHESS) {
            sp::ChessRules rules;
            analyse_emul(rules, &sp::chess_tables(), cfg, n, fens, moves, offsets, n_slots, pool_words, depth, roots_cap, f, nullptr, r->res);
        } else {
            sp::TttRules rules;
            analyse_emul(rules, &rules, cfg, n, fens, moves, offsets, n_slots, pool_words, depth, roots_cap, f, nullptr, r->res);
        }
    } catch (const sp::SpError& e) {
        r->error = e.msg.empty() ? "error" : e.msg;
    }
    return r.release();
}
const char* analysis_emul_error(void* h) { return static_cast<AnalysisEmulResult*>(h)->error.c_str(); }
int analysis_emul_count(const void* h, uint32_t* n) {
    *n = static_cast<uint32_t>(static_cast<const AnalysisEmulResult*>(h)->res.size());
    return 0;
}
int analysis_emul_get(const void* h, uint32_t k, cattus_b200_analysis_position* out) {
    return ds::analysis_get(static_cast<const AnalysisEmulResult*>(h)->res, k, out);
}
int analysis_emul_children(const void* h, uint32_t k, uint16_t* moves, uint32_t* visits, float* w, float* priors, uint32_t cap) {
    return ds::analysis_children(static_cast<const AnalysisEmulResult*>(h)->res, k, moves, visits, w, priors, cap);
}
int analysis_emul_pv(const void* h, uint32_t k, uint16_t* pv, uint32_t cap) { return ds::analysis_pv(static_cast<const AnalysisEmulResult*>(h)->res, k, pv, cap); }
void analysis_emul_free(void* h) { delete static_cast<AnalysisEmulResult*>(h); }
}
