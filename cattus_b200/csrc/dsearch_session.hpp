// Host half of a persistent device search session (include/cattus_b200_session.h, DESIGN.md section 17).
//
// A session is one slot of the device-resident search that keeps its tree across searches.  Each search is a run of waves
// of the minibatch kernels: the first wave's begin (Core::begin_slot<true>) installs the position's history with
// kCmdSetRoot | kCmdKeepTree and keeps the subtree of the new root when the old tree has it; every wave after that runs
// one minibatch.  The device ends the search at a minibatch boundary -- node budget, minibatch cap, the stop word, tree
// capacity -- and posts the analysis entry with the minibatch / collision counts, the kept visits and the reason.  The
// host thread of the session submits the waves, keeps depth() of them in flight, and writes the stop word when the
// deadline passes on its steady clock.
//
// `Backend` is DsCudaBackend (dsearch.cuh) built with a session, or the emulation in tests/emul: one slot, the analysis
// result layout with minibatch counts, a root upload, and session_ctl() / snapshot() in memory the device reads and
// writes while the host does.
#pragma once

#include <chrono>
#include <condition_variable>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/cattus_b200_session.h"
#include "dsearch_analysis.hpp"

namespace ds {

// Type-erased session: the C ABI holds one of these whatever the game.
class SessionBase {
  public:
    virtual ~SessionBase() = default;
    virtual void set_position(const char* fen, const uint16_t* moves, uint32_t n) = 0;
    virtual void new_game() = 0;
    virtual void go(const cattus_b200_session_limits& limits) = 0;
    virtual void stop() = 0;
    virtual void info(cattus_b200_session_snapshot& out) = 0;
    // false: still running after timeout_ms; true: `out` holds the result (or the search's error is thrown)
    virtual bool wait(uint32_t timeout_ms, std::vector<AnalysisResult>& out) = 0;
};

// L of a session's options
inline uint32_t session_search_batch(const cattus_b200_session_opts* opts, uint32_t max_batch) {
    if (!opts || opts->struct_size != sizeof(cattus_b200_session_opts)) throw sp::SpError{CATTUS_B200_EINVAL, "session opts struct_size mismatch"};
    if (opts->search_batch < 2) throw sp::SpError{CATTUS_B200_EINVAL, "session: search_batch must be >= 2 (a session searches in minibatches)"};
    if (opts->search_batch > max_batch)
        throw sp::SpError{CATTUS_B200_EINVAL, "session: search_batch (" + std::to_string(opts->search_batch) + ") exceeds the evaluator's max_batch (" +
                                                  std::to_string(max_batch) + ")"};
    return opts->search_batch;
}

// Words of each of a session's tree buffers: tree_kwords x 1024, or the largest the 2^26-word tree address space allows
// (edges hold a child's block offset / 4 + 1 in 24 bits).  It must hold a few minibatches' worth of new leaves.
inline uint32_t session_tree_words(uint32_t tree_kwords, unsigned long long minibatch_words) {
    const unsigned long long limit = (static_cast<unsigned long long>(0xFFFFFE) << 2) - 4u;
    const unsigned long long want = tree_kwords ? static_cast<unsigned long long>(tree_kwords) * 1024u : limit;
    if (want > limit) throw sp::SpError{CATTUS_B200_EINVAL, "session: tree_kwords beyond the 2^26-word tree address space"};
    if (want < 4u * minibatch_words)
        throw sp::SpError{CATTUS_B200_EINVAL, "session: tree_kwords must hold at least 4 minibatches of new leaves (" +
                                                  std::to_string((4u * minibatch_words + 1023u) / 1024u) + " kwords)"};
    return static_cast<uint32_t>(want & ~3ull);
}

template <class Rules, class Backend>
class SessionDriver final : public SessionBase {
    using Pos = typename Rules::Pos;
    using Move = typename Rules::Move;
    using Clock = std::chrono::steady_clock;

  public:
    // params: the analysis parameters (sim_num is not used: each search has its own budget)
    SessionDriver(const Rules& rules, const sp::Params& params, std::unique_ptr<Backend> be, uint32_t search_batch)
        : R(rules), params_(params), be_(std::move(be)), search_batch_(search_batch) {
        result_stride_ = analysis_stride_for(be_->max_children(), search_batch_);
        cmd_stride_ = cmd_stride_for(be_->max_children());
    }
    ~SessionDriver() override {
        stop();
        if (thread_.joinable()) thread_.join();
    }

    void set_position(const char* fen, const uint16_t* moves, uint32_t n) override {
        std::lock_guard<std::mutex> g(mu_);
        if (running_) throw sp::SpError{CATTUS_B200_EINVAL, "session: set_position while a search runs"};
        const uint32_t offsets[2] = {0, n};
        const char* fens[1] = {fen};
        hist_ = analysis_histories(R, 1, fens, moves, offsets, "position")[0];
        has_position_ = true;
    }

    void new_game() override {
        std::lock_guard<std::mutex> g(mu_);
        if (running_) throw sp::SpError{CATTUS_B200_EINVAL, "session: new_game while a search runs"};
        keep_tree_ = false;
    }

    void go(const cattus_b200_session_limits& lim) override {
        std::unique_lock<std::mutex> g(mu_);
        if (lim.struct_size != sizeof(cattus_b200_session_limits)) throw sp::SpError{CATTUS_B200_EINVAL, "session limits struct_size mismatch"};
        if (running_) throw sp::SpError{CATTUS_B200_EINVAL, "session: go while a search runs"};
        if (!has_position_) throw sp::SpError{CATTUS_B200_EINVAL, "session: go before set_position"};
        if (thread_.joinable()) thread_.join();
        volatile SessionCtl* c = be_->session_ctl();
        c->nodes = lim.nodes ? lim.nodes : 0xFFFFFFFFu;
        c->max_minibatches = lim.minibatches ? lim.minibatches : 0xFFFFFFFFu;
        c->stop = kStopNone;
        c->info = 0;
        snap_seq0_ = snapshot_seq();
        t0_ = Clock::now();
        has_deadline_ = lim.deadline_us != 0;
        deadline_ = t0_ + std::chrono::microseconds(lim.deadline_us);
        result_.assign(1, AnalysisResult());
        error_code_ = 0;
        error_.clear();
        root_ = hist_.back();
        const int st = analysis_root_status(R, hist_);
        if (st != 0) {  // the game is over: no search, the tree stays as it is
            result_[0].status = static_cast<uint32_t>(st);
            result_[0].stop_reason = CATTUS_B200_STOP_FINISHED;
            t_end_ = t0_;
            done_ = true;
            return;
        }
        running_ = true;
        done_ = false;
        thread_ = std::thread([this] { run(); });
    }

    void stop() override {
        std::lock_guard<std::mutex> g(mu_);
        if (running_ && be_->session_ctl()->stop == kStopNone) be_->session_ctl()->stop = kStopRequest;
    }

    void info(cattus_b200_session_snapshot& out) override {
        std::lock_guard<std::mutex> g(mu_);
        const uint32_t size = out.struct_size;
        std::memset(&out, 0, sizeof(out));
        out.struct_size = size;
        out.searching = running_ ? 1u : 0u;
        out.seconds = std::chrono::duration<double>((running_ ? Clock::now() : t_end_) - t0_).count();
        if (running_) be_->session_ctl()->info = 1;
        // seqlock: an even sequence word, the same before and after the copy
        const uint8_t* snap = be_->snapshot();
        std::vector<uint8_t> buf(kSnapshotHdr + result_stride_);
        bool ok = false;
        for (int tries = 0; tries < 8 && !ok; ++tries) {
            const uint32_t s1 = snapshot_seq();
            if (s1 & 1u) {
                std::this_thread::yield();
                continue;
            }
            __atomic_thread_fence(__ATOMIC_ACQUIRE);
            std::memcpy(buf.data(), snap, buf.size());
            __atomic_thread_fence(__ATOMIC_ACQUIRE);
            ok = snapshot_seq() == s1;
            if (ok && s1 == snap_seq0_) return;  // nothing of this search yet
        }
        if (!ok) return;
        const uint32_t* hdr = reinterpret_cast<const uint32_t*>(buf.data());
        const uint8_t* e = buf.data() + kSnapshotHdr;
        const AnalysisHdr* ah = reinterpret_cast<const AnalysisHdr*>(e);
        if (ah->count == 0 || ah->count > be_->max_children() || ah->pv_len > kPvMax) return;  // the root is not expanded yet
        AnalysisResult r;
        read_analysis_entry(R, params_, root_, e, be_->max_children(), result_stride_, search_batch_, r, probs_info_, weights_info_);
        out.valid = 1;
        out.simulations = hdr[1];
        out.minibatches = hdr[2];
        out.collisions = hdr[3];
        out.best_move = r.best;
        out.q = r.q;
        out.pv_len = static_cast<uint16_t>(r.pv.size());
        for (size_t i = 0; i < r.pv.size(); ++i) out.pv[i] = r.pv[i];
    }

    bool wait(uint32_t timeout_ms, std::vector<AnalysisResult>& out) override {
        std::unique_lock<std::mutex> g(mu_);
        if (!done_ && !running_) throw sp::SpError{CATTUS_B200_EINVAL, "session: wait without a search"};
        const auto ready = [this] { return done_; };
        if (timeout_ms == 0xFFFFFFFFu)
            cv_.wait(g, ready);
        else if (!cv_.wait_for(g, std::chrono::milliseconds(timeout_ms), ready))
            return false;
        if (error_code_) throw sp::SpError{error_code_, error_};
        out = result_;
        return true;
    }

  private:
    uint32_t snapshot_seq() const { return *reinterpret_cast<const volatile uint32_t*>(be_->snapshot()); }

    void run() {
        int code = 0;
        std::string msg;
        try {
            be_->bind_thread();
            if (failed_) {  // the last search met a device error: its error word and virtual counts go, the tree is dropped
                be_->clear_error();
                failed_ = false;
            }
            search();
        } catch (const sp::SpError& e) {
            code = e.code ? e.code : CATTUS_B200_EDEVICE;
            msg = e.msg;
        } catch (const std::exception& e) {
            code = be_->error_code(e);
            msg = e.what();
        }
        std::lock_guard<std::mutex> g(mu_);
        t_end_ = Clock::now();
        result_[0].seconds = std::chrono::duration<double>(t_end_ - t0_).count();
        if (code) {
            error_code_ = code;
            error_ = msg;
            keep_tree_ = false;  // the device tree is in an unknown state
            failed_ = true;
        }
        running_ = false;
        done_ = true;
        cv_.notify_all();
    }

    // The waves of one search: the first carries the begin command, the rest run a minibatch each, until a wave posts the
    // result; the waves still in flight then find the slot done and are drained.
    void search() {
        const uint32_t depth = std::max<uint32_t>(1, be_->depth());
        const uint32_t len = static_cast<uint32_t>(hist_.size());
        if (len > be_->roots_cap()) throw sp::SpError{CATTUS_B200_EINVAL, "session: history longer than the root upload"};
        std::deque<uint32_t> inflight;
        bool first = true, finished = false;
        volatile SessionCtl* c = be_->session_ctl();
        while (!finished || !inflight.empty()) {
            if (!finished && inflight.size() < depth) {
                const uint32_t w = wave_++;
                uint8_t* block = be_->cmd_block(w);
                uint32_t* hdr = reinterpret_cast<uint32_t*>(block);
                uint32_t n_cmds = 0, n_roots = 0;
                if (first) {
                    std::copy(hist_.begin(), hist_.end(), be_->roots_block(w));
                    Cmd cmd;
                    std::memset(&cmd, 0, sizeof(cmd));
                    cmd.slot = 0;
                    cmd.flags = kCmdSetRoot | (keep_tree_ ? kCmdKeepTree : 0u);
                    cmd.root_at = 0;
                    cmd.root_len = len;
                    std::memset(block + 16, 0, cmd_stride_);
                    std::memcpy(block + 16, &cmd, sizeof(cmd));
                    n_cmds = 1;
                    n_roots = len;
                    first = false;
                }
                hdr[0] = n_cmds;
                hdr[1] = w;
                hdr[2] = hdr[3] = 0;
                be_->submit(w, 0, n_cmds, n_roots);
                inflight.push_back(w);
                continue;
            }
            if (has_deadline_ && c->stop == kStopNone && Clock::now() >= deadline_) c->stop = kStopDeadline;
            const uint32_t w = inflight.front();
            inflight.pop_front();
            uint32_t n_done = 0;
            const uint8_t* res = be_->wait(w, &n_done);
            if (n_done) {
                on_result(res);
                finished = true;
            }
        }
        keep_tree_ = true;
    }

    void on_result(const uint8_t* e) {
        const AnalysisHdr* ah = reinterpret_cast<const AnalysisHdr*>(e);
        if (ah->slot != 0 || ah->count > be_->max_children() || ah->count == 0 || ah->pv_len > kPvMax)
            throw sp::SpError{CATTUS_B200_EDEVICE, "device search posted a malformed result"};
        std::lock_guard<std::mutex> g(mu_);
        AnalysisResult& r = result_[0];
        read_analysis_entry(R, params_, root_, e, be_->max_children(), result_stride_, search_batch_, r, probs_, weights_);
        const uint32_t* counts = reinterpret_cast<const uint32_t*>(e + result_stride_ - 16u);
        r.reused = counts[2];
        r.stop_reason = counts[3];
        // the final minibatch also posted the snapshot: its simulation count is this search's
        r.simulations = reinterpret_cast<const uint32_t*>(be_->snapshot())[1];
    }

    const Rules R;
    const sp::Params params_;
    std::unique_ptr<Backend> be_;
    const uint32_t search_batch_;
    uint32_t result_stride_ = 0, cmd_stride_ = 0, wave_ = 0, snap_seq0_ = 0;
    std::vector<Pos> hist_;
    Pos root_{};
    bool has_position_ = false, keep_tree_ = false, running_ = false, done_ = false, has_deadline_ = false, failed_ = false;
    Clock::time_point t0_{}, t_end_{}, deadline_{};
    std::vector<AnalysisResult> result_;
    int error_code_ = 0;
    std::string error_;
    std::mutex mu_;
    std::condition_variable cv_;
    std::thread thread_;
    std::vector<std::pair<Move, float>> probs_, probs_info_;
    std::vector<float> weights_, weights_info_;
};

// ---------------------------------------------------------------- entry points shared by the C ABI and the test emulation
inline int session_stats(const std::vector<AnalysisResult>& r, cattus_b200_session_stats* out) {
    if (!out || r.size() != 1) return CATTUS_B200_EINVAL;
    if (out->struct_size != sizeof(cattus_b200_session_stats)) return CATTUS_B200_EINVAL;
    out->stop_reason = r[0].stop_reason;
    out->reused_visits = r[0].reused;
    out->pad = 0;
    out->seconds = r[0].seconds;
    return CATTUS_B200_OK;
}

}  // namespace ds
