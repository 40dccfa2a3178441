// TEST INFRASTRUCTURE -- never part of the product library.
//
// Self-play and match play with minibatches under virtual loss per side (DESIGN.md section 16) over the host emulation
// of the device-resident search: match_emul.cpp's backend (self-play result layout, root upload) with an evaluator batch
// of n_slots x the larger search_batch rows per evaluator, the per-descent buffers, the virtual counts and the minibatch
// kernels' per-slot code.  With search_batch 1 on both sides it runs the one-leaf code unchanged, as the CUDA backend
// does.  The CPU tests compare it with tests/batch_game_oracle.py's game loop over BatchedPlayer.
#include "match_emul.cpp"

namespace {

template <class Rules>
struct EmulSideBatchBackend : EmulMatchBackend<Rules> {
    using Base = EmulMatchBackend<Rules>;
    uint32_t Lmax;
    std::vector<ds::BatchDescent> descents;
    std::vector<ds::PathStep> bpaths;
    std::vector<uint32_t> vcount;

    EmulSideBatchBackend(const Rules& rules, const void* blob, uint32_t n_slots, uint32_t pool_words, uint32_t depth, const sp::Params params[2],
                         cattus_b200_eval_fn f1, cattus_b200_eval_fn f2, uint32_t cache_size, uint32_t roots_cap, const uint32_t search_batch[2])
        : Base(rules, blob, n_slots, pool_words, depth, params, f1, f2, cache_size, roots_cap),
          Lmax(std::max(search_batch[0], search_batch[1])) {
        if (Lmax <= 1) return;
        if (this->n_pops != 1) throw sp::SpError{CATTUS_B200_EINVAL, "emul: minibatches run one population"};
        ds::Params<Rules>& p = this->p;
        const uint32_t rows = n_slots * Lmax;
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
        descents.assign(static_cast<size_t>(n_slots) * Lmax, ds::BatchDescent{});
        bpaths.resize(static_cast<size_t>(n_slots) * Lmax * p.path_cap);
        vcount.assign(static_cast<size_t>(n_slots) * (pool_words >> 2), 0u);
        p.search_batch.side[0] = std::max<uint32_t>(1, search_batch[0]);
        p.search_batch.side[1] = std::max<uint32_t>(1, search_batch[1]);
        p.search_batch.max = Lmax;
        p.descents = descents.data();
        p.bpaths = bpaths.data();
        p.vcount = vcount.data();
    }

    void submit(uint32_t wave, uint32_t pop, uint32_t n_cmds, uint32_t n_roots) {
        if (Lmax <= 1) {
            Base::submit(wave, pop, n_cmds, n_roots);
            return;
        }
        ds::Params<Rules>& p = this->p;
        this->done_count = 0;
        *p.eval[0].n_ptr = 0;
        *p.eval[1].n_ptr = 0;
        decltype(auto) rules = ds::RulesRef<Rules>::get(p.rules);
        // the invariant tree reuse relies on: a slot that begins a search (and may move its tree) holds no virtual count
        const uint32_t units = (p.pool_words >> 2);
        for (uint32_t ci = 0; ci < n_cmds; ++ci) {
            const ds::Cmd* c = reinterpret_cast<const ds::Cmd*>(p.cmds + 16 + static_cast<size_t>(ci) * p.cmd_stride);
            for (uint32_t u = 0; u < units; ++u)
                if (vcount[static_cast<size_t>(c->slot) * units + u]) throw sp::SpError{CATTUS_B200_EDEVICE, "emul: a virtual count outlived its minibatch"};
        }
        if (!p.begin_lead)
            for (uint32_t ci = 0; ci < n_cmds; ++ci) ds::Core<Rules>::begin_slot(rules, p, ci, wave);
        for (uint32_t si = 0; si < p.n_slots; ++si) ds::Core<Rules>::batch_select_slot(rules, p, si, wave);
        if (p.begin_lead)
            for (uint32_t ci = 0; ci < n_cmds; ++ci) ds::Core<Rules>::begin_slot(rules, p, ci, wave);
        for (uint32_t e = 0; e < p.n_evals; ++e) this->run_eval(p, this->probs, this->values, static_cast<int>(e));
        for (uint32_t si = 0; si < p.n_slots; ++si) ds::Core<Rules>::batch_expand_slot(rules, p, si, wave);
        this->done_per_buf[wave % this->n_bufs] = this->done_count;
    }
};

template <class Rules>
void selfplay_batch(const Rules& rules, const void* blob, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_selfplay_opts* opts, uint32_t max_batch,
                    uint32_t pool_words, uint32_t depth, cattus_b200_eval_fn f1, cattus_b200_eval_fn f2, sp::Shared& sh) {
    const uint32_t L = sp::selfplay_search_batch(opts, *cfg);
    const uint32_t search_batch[2] = {L, L};
    const sp::Params p = sp::parse_params(cfg);
    const sp::Params params[2] = {p, p};
    const uint32_t stride = std::max<uint32_t>(1, cfg->game_stride);
    const uint32_t games = cfg->games_num > cfg->first_game ? (cfg->games_num - cfg->first_game + stride - 1) / stride : 0;
    if (games == 0) return;
    const uint32_t n_slots = ds::selfplay_slots(cfg->device_games, games, max_batch, L);
    EmulSideBatchBackend<Rules> be(rules, blob, n_slots, pool_words, depth, params, f1, f2, cfg->cache_size, ds::hist_cap_for<Rules>(), search_batch);
    ds::Driver<Rules, EmulSideBatchBackend<Rules>> drv(rules, *cfg, params, be, sh, nullptr, search_batch);
    drv.run();
}

template <class Rules>
void match_batch(const Rules& rules, const void* blob, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_match_side* side_b,
                 const cattus_b200_match_opts* opts, uint32_t max_batch, uint32_t n, const char* const* fens, const uint16_t* moves,
                 const uint32_t* offsets, uint32_t pool_words, uint32_t depth, uint32_t roots_cap, cattus_b200_eval_fn fa, cattus_b200_eval_fn fb,
                 ds::MatchResult& out) {
    uint32_t search_batch[2];
    ds::match_search_batch(opts, search_batch);
    sp::Params params[2];
    ds::match_params(*cfg, side_b, params);
    const auto openings = ds::match_openings(rules, n, fens, moves, offsets, out.opening_status);
    const uint32_t games = ds::match_games(out.opening_status);
    if (!games) return;
    const uint32_t n_slots = ds::analysis_slots(cfg->device_games, games, max_batch, std::max(search_batch[0], search_batch[1]));
    EmulSideBatchBackend<Rules> be(rules, blob, n_slots, pool_words, depth, params, fa, fb, cfg->cache_size,
                                   std::max(roots_cap, ds::hist_cap_for<Rules>()), search_batch);
    ds::match_play(rules, *cfg, params, be, openings, out, search_batch);
}

template <class F>
void for_game(const cattus_b200_selfplay_cfg* cfg, F&& f) {
    if (cfg->game == CATTUS_B200_GAME_HEX) {
        if (cfg->board_size <= 8) {
            sp::HexRulesT<uint64_t> rules(static_cast<int>(cfg->board_size));
            f(rules, &rules);
        } else {
            sp::HexRulesT<sp::u128> rules(static_cast<int>(cfg->board_size));
            f(rules, &rules);
        }
    } else if (cfg->game == CATTUS_B200_GAME_CHESS) {
        sp::ChessRules rules;
        f(rules, static_cast<const void*>(&sp::chess_tables()));
    } else {
        sp::TttRules rules;
        f(rules, &rules);
    }
}

}  // namespace

extern "C" {

// Self-play as cattus_b200_selfplay_run_opts plays it: opts NULL is one leaf in flight; f2 NULL: one evaluator (one
// handle); max_batch: the evaluator batch the slots are checked against (cfg->device_games slots at most); depth: the
// test knobs of dsearch_emul_run.  Read the result with dsearch_emul_*; *code is the error code.
void* selfplay_batch_emul_run(cattus_b200_eval_fn f1, cattus_b200_eval_fn f2, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_selfplay_opts* opts,
                              uint32_t max_batch, uint32_t pool_words, uint32_t depth, int* code) {
    std::unique_ptr<EmulResult> r(new EmulResult());
    *code = 0;
    try {
        for_game(cfg, [&](const auto& rules, const void* blob) { selfplay_batch(rules, blob, cfg, opts, max_batch, pool_words, depth, f1, f2, r->sh); });
    } catch (const sp::SpError& e) {
        r->error = e.msg.empty() ? "error" : e.msg;
        *code = e.code;
    }
    std::sort(r->sh.records.begin(), r->sh.records.end(), [](const sp::GameRecord& a, const sp::GameRecord& b) { return a.game_idx < b.game_idx; });
    return r.release();
}
// per model (1, 2): out[0..1] minibatches, out[2..3] collisions
void selfplay_batch_emul_batches(void* h, uint64_t out[4]) {
    const sp::Shared& s = static_cast<EmulResult*>(h)->sh;
    out[0] = s.minibatches[0];
    out[1] = s.minibatches[1];
    out[2] = s.collisions[0];
    out[3] = s.collisions[1];
}

// A match as cattus_b200_match_run_opts plays it (fb NULL: one evaluator); read it with match_emul_*.
void* match_batch_emul_run(cattus_b200_eval_fn fa, cattus_b200_eval_fn fb, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_match_side* side_b,
                           const cattus_b200_match_opts* opts, uint32_t max_batch, uint32_t n, const char* const* fens, const uint16_t* moves,
                           const uint32_t* offsets, uint32_t pool_words, uint32_t depth, uint32_t roots_cap, int* code) {
    std::unique_ptr<MatchEmulResult> r(new MatchEmulResult());
    *code = 0;
    try {
        for_game(cfg, [&](const auto& rules, const void* blob) {
            match_batch(rules, blob, cfg, side_b, opts, max_batch, n, fens, moves, offsets, pool_words, depth, roots_cap, fa, fb, r->res);
        });
    } catch (const sp::SpError& e) {
        r->error = e.msg.empty() ? "error" : e.msg;
        *code = e.code;
    }
    return r.release();
}
int match_batch_emul_batches(const void* h, uint32_t side, uint64_t* minibatches, uint64_t* collisions) {
    return ds::match_batches(static_cast<const MatchEmulResult*>(h)->res, side, minibatches, collisions);
}
}
