// TEST INFRASTRUCTURE -- never part of the product library.
//
// Persistent search sessions (cattus_b200/csrc/dsearch_session.hpp, DESIGN.md section 17) over the host emulation of the
// device-resident search: search_batch_emul.cpp's minibatch backend with one slot, the session's begin
// (Core::begin_slot<true>), its control words and its snapshot.  The same SessionDriver as the library runs it, host thread
// included.  The CPU tests compare it with tests/session_oracle.py.
#include "search_batch_emul.cpp"

#include "../../cattus_b200/csrc/dsearch_session.hpp"

namespace {

template <class Rules>
struct EmulSessionBackend : EmulBatchBackend<Rules> {
    using Base = EmulBatchBackend<Rules>;
    ds::SessionCtl ctl{};
    std::vector<uint8_t> snap;
    uint32_t stop_after = 0, waves_seen = 0;

    // stop_after > 0: the backend writes the stop word itself once that many waves have run (a stop at a known wave)
    EmulSessionBackend(const Rules& rules, const void* blob, uint32_t pool_words, uint32_t depth, const sp::Params params[2], cattus_b200_eval_fn f,
                       uint32_t cache_size, uint32_t search_batch, uint32_t stop_after_waves)
        : Base(rules, blob, 1, pool_words, depth & 0xFFu, params, f, cache_size, ds::hist_cap_for<Rules>(), search_batch), stop_after(stop_after_waves) {
        ds::Params<Rules>& p = this->p;
        snap.assign(ds::kSnapshotHdr + p.result_stride, 0);
        p.session = &ctl;
        p.snapshot = snap.data();
        p.sim_num[0] = p.sim_num[1] = 0;
        p.begin_lead = 0;
    }
    volatile ds::SessionCtl* session_ctl() { return &ctl; }
    const uint8_t* snapshot() const { return snap.data(); }
    void bind_thread() {}
    void clear_error() {
        this->error = 0;
        std::fill(this->vcount.begin(), this->vcount.end(), 0u);
    }
    int error_code(const std::exception&) const { return CATTUS_B200_EDEVICE; }

    void submit(uint32_t wave, uint32_t, uint32_t n_cmds, uint32_t) {
        ds::Params<Rules>& p = this->p;
        this->done_count = 0;
        *p.eval[0].n_ptr = 0;
        *p.eval[1].n_ptr = 0;
        decltype(auto) rules = ds::RulesRef<Rules>::get(p.rules);
        for (uint32_t ci = 0; ci < n_cmds; ++ci) ds::Core<Rules>::template begin_slot<true>(rules, p, ci, wave);
        ds::Core<Rules>::batch_select_slot(rules, p, 0, wave);
        // the device evaluator runs at most its batch of rows; the row counter may have run past it (kErrRows)
        *p.eval[0].n_ptr = std::min(*p.eval[0].n_ptr, p.eval[0].max_rows);
        this->run_eval(p, this->probs, this->values, 0);
        ds::Core<Rules>::batch_expand_slot(rules, p, 0, wave);
        this->done_per_buf[wave % this->n_bufs] = this->done_count;
        if (stop_after && ++waves_seen == stop_after) ctl.stop = ds::kStopRequest;
    }
};

template <class Rules>
std::unique_ptr<ds::SessionBase> make_session(const Rules& rules, const void* blob, const cattus_b200_selfplay_cfg& cfg, const cattus_b200_session_opts* opts,
                                              uint32_t max_batch, uint32_t depth, uint32_t stop_after, cattus_b200_eval_fn f, uint32_t** max_rows) {
    cattus_b200_selfplay_cfg c = cfg;
    c.sim_num = std::max<uint32_t>(c.sim_num, 2u);
    const sp::Params params[2] = {ds::analysis_params(c), ds::analysis_params(c)};
    const uint32_t L = ds::session_search_batch(opts, max_batch);
    using T = ds::TreeOps<Rules>;
    const uint32_t maxc = Rules::kChess ? 224u : static_cast<uint32_t>(rules.max_children());
    const uint32_t words = ds::session_tree_words(opts->tree_kwords, static_cast<unsigned long long>(L) * T::block_words(static_cast<int>(maxc)));
    std::unique_ptr<EmulSessionBackend<Rules>> be(new EmulSessionBackend<Rules>(rules, blob, words, depth, params, f, cfg.cache_size, L, stop_after));
    *max_rows = &be->p.eval[0].max_rows;
    return std::unique_ptr<ds::SessionBase>(new ds::SessionDriver<Rules, EmulSessionBackend<Rules>>(rules, params[0], std::move(be), L));
}

// the rule object of a game lives as long as the session (hex tables are read in place through the blob pointer)
struct RulesHolder {
    std::unique_ptr<sp::HexRulesT<uint64_t>> hex;
    std::unique_ptr<sp::HexRulesT<sp::u128>> hex_big;
    sp::TttRules ttt;
    sp::ChessRules chess;
};

struct SessionEmulHandle {
    RulesHolder rules;
    std::unique_ptr<ds::SessionBase> s;
    uint32_t* max_rows = nullptr;  // the evaluator batch the device may fill (a smaller one makes a minibatch fail with kErrRows)
};

thread_local std::string g_error;

template <class F>
int guarded(F&& f) {
    try {
        f();
        g_error.clear();
        return 0;
    } catch (const sp::SpError& e) {
        g_error = e.msg;
        return e.code ? e.code : CATTUS_B200_EINVAL;
    }
}

}  // namespace

extern "C" {

// max_batch: the evaluator batch L is checked against; depth: waves in flight; stop_after_waves: see EmulSessionBackend.
// The tree buffer is opts->tree_kwords (0: the 2^26-word maximum).
int session_emul_create(cattus_b200_eval_fn f, const cattus_b200_selfplay_cfg* cfg, const cattus_b200_session_opts* opts, uint32_t max_batch, uint32_t depth,
                        uint32_t stop_after_waves, void** out) {
    return guarded([&] {
        std::unique_ptr<SessionEmulHandle> h(new SessionEmulHandle());
        if (cfg->struct_size != sizeof(cattus_b200_selfplay_cfg)) throw sp::SpError{CATTUS_B200_EINVAL, "selfplay cfg struct_size mismatch"};
        if (cfg->game == CATTUS_B200_GAME_HEX) {
            if (cfg->board_size <= 8) {
                h->rules.hex.reset(new sp::HexRulesT<uint64_t>(static_cast<int>(cfg->board_size)));
                h->s = make_session(*h->rules.hex, h->rules.hex.get(), *cfg, opts, max_batch, depth, stop_after_waves, f, &h->max_rows);
            } else {
                h->rules.hex_big.reset(new sp::HexRulesT<sp::u128>(static_cast<int>(cfg->board_size)));
                h->s = make_session(*h->rules.hex_big, h->rules.hex_big.get(), *cfg, opts, max_batch, depth, stop_after_waves, f, &h->max_rows);
            }
        } else if (cfg->game == CATTUS_B200_GAME_CHESS) {
            h->s = make_session(h->rules.chess, &sp::chess_tables(), *cfg, opts, max_batch, depth, stop_after_waves, f, &h->max_rows);
        } else {
            h->s = make_session(h->rules.ttt, &h->rules.ttt, *cfg, opts, max_batch, depth, stop_after_waves, f, &h->max_rows);
        }
        *out = h.release();
    });
}
const char* session_emul_last_error() { return g_error.c_str(); }
int session_emul_set_position(void* h, const char* fen, const uint16_t* moves, uint32_t n) {
    return guarded([&] { static_cast<SessionEmulHandle*>(h)->s->set_position(fen, moves, n); });
}
int session_emul_new_game(void* h) {
    return guarded([&] { static_cast<SessionEmulHandle*>(h)->s->new_game(); });
}
int session_emul_go(void* h, const cattus_b200_session_limits* lim) {
    return guarded([&] { static_cast<SessionEmulHandle*>(h)->s->go(*lim); });
}
int session_emul_stop(void* h) {
    return guarded([&] { static_cast<SessionEmulHandle*>(h)->s->stop(); });
}
int session_emul_info(void* h, cattus_b200_session_snapshot* out) {
    return guarded([&] {
        if (out->struct_size != sizeof(cattus_b200_session_snapshot)) throw sp::SpError{CATTUS_B200_EINVAL, "session snapshot struct_size mismatch"};
        static_cast<SessionEmulHandle*>(h)->s->info(*out);
    });
}
// result: an AnalysisEmulResult (analysis_emul_* accessors)
int session_emul_wait(void* h, uint32_t timeout_ms, void** result) {
    std::unique_ptr<AnalysisEmulResult> r(new AnalysisEmulResult());
    bool done = false;
    const int rc = guarded([&] { done = static_cast<SessionEmulHandle*>(h)->s->wait(timeout_ms, r->res); });
    if (rc) return rc;
    if (!done) return CATTUS_B200_SESSION_RUNNING;
    *result = r.release();
    return 0;
}
int session_emul_batches(const void* r, uint32_t k, uint32_t* minibatches, uint32_t* collisions) {
    return ds::analysis_batches(static_cast<const AnalysisEmulResult*>(r)->res, k, minibatches, collisions);
}
int session_emul_result_stats(const void* r, cattus_b200_session_stats* out) { return ds::session_stats(static_cast<const AnalysisEmulResult*>(r)->res, out); }
// rows: the evaluator rows a minibatch may write from the next search on (between searches only)
void session_emul_set_max_rows(void* h, uint32_t rows) { *static_cast<SessionEmulHandle*>(h)->max_rows = rows; }
void session_emul_destroy(void* h) { delete static_cast<SessionEmulHandle*>(h); }
}
