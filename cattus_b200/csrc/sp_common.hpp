// Pieces of the self-play driver shared by its two arrangements: trees on the host (csrc/selfplay.cpp) and trees in HBM
// (csrc/dsearch_host.hpp).  Everything here is the GAME side of the reference's self-play loop
// (training/self-play/src/self_play.rs:179-276): the per-game random stream, MctsParams, the move choice of
// MctsPlayer::choose_move_from_probabilities (engine/src/mcts/mod.rs:387-417), the Dirichlet draw of
// add_dirichlet_noise (mod.rs:419-446) and the .traindata serializers (self_play.rs:33-61, serialize/hex.rs:16-28,
// serialize/ttt.rs:17-22, serialize/chess.rs:18-57).
#pragma once

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../../include/cattus_b200_selfplay.h"
#include "chess_rules.hpp"
#include "sp_rules.hpp"

namespace sp {

using Clock = std::chrono::steady_clock;

struct SpError {
    int code;
    std::string msg;
};

// ------------------------------------------------------------------------------------------------ random stream
// The reference uses the unseeded thread-local rand::rng(); every game here owns this stream instead (same
// definition in oracle/mcts.py so whole games can be compared).
struct SplitMix64 {
    uint64_t state;
    explicit SplitMix64(uint64_t seed = 0) : state(seed) {}
    uint64_t next_u64() {
        state += 0x9E3779B97F4A7C15ull;
        uint64_t z = state;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    }
    double next_f64() { return static_cast<double>(next_u64() >> 11) * (1.0 / 9007199254740992.0); }
    double next_open_f64() { return (static_cast<double>(next_u64() >> 12) + 0.5) * (1.0 / 4503599627370496.0); }
    double normal() {
        const double u1 = next_open_f64();
        const double u2 = next_f64();
        return std::sqrt(-2.0 * std::log(u1)) * std::cos(2.0 * M_PI * u2);
    }
    double gamma(double alpha) {  // Marsaglia-Tsang; alpha < 1 boosted with U^(1/alpha)
        if (alpha < 1.0) {
            const double u = next_open_f64();
            return gamma(alpha + 1.0) * std::pow(u, 1.0 / alpha);
        }
        const double d = alpha - 1.0 / 3.0;
        const double c = 1.0 / std::sqrt(9.0 * d);
        for (;;) {
            const double x = normal();
            double v = 1.0 + c * x;
            if (v <= 0.0) continue;
            v = v * v * v;
            const double u = next_open_f64();
            if (std::log(u) < 0.5 * x * x + d - d * v + d * std::log(v)) return d * v;
        }
    }
};

static inline uint64_t game_seed(uint64_t base, uint32_t game_idx) { return base ^ (0xD1B54A32D192ED03ull * (static_cast<uint64_t>(game_idx) + 1)); }

struct Params {
    uint32_t sim_num;
    float explore_factor;
    std::vector<std::pair<uint32_t, float>> temperatures;
    float last_temperature;
    float noise_alpha, noise_eps;
    float temperature_at(size_t move_num) const {  // TemperaturePolicy::get_temperature, mod.rs:482-488
        for (auto& t : temperatures)
            if (move_num < t.first) return t.second;
        return last_temperature;
    }
};

// MctsParams from the config (mcts/mod.rs:72-110; TemperaturePolicy::scheduled, self_play_cmd.rs:68-72)
inline Params parse_params(const cattus_b200_selfplay_cfg* cfg) {
    if (cfg->sim_num < 2) throw SpError{CATTUS_B200_EINVAL, "sim_num must be > 1 (mcts/mod.rs:157)"};
    if (!(cfg->explore_factor >= 0.0f) || !(cfg->prior_noise_alpha >= 0.0f) || !(cfg->prior_noise_epsilon >= 0.0f && cfg->prior_noise_epsilon <= 1.0f))
        throw SpError{CATTUS_B200_EINVAL, "bad mcts parameters (mcts/mod.rs:107-110)"};
    Params p;
    p.sim_num = cfg->sim_num;
    p.explore_factor = cfg->explore_factor;
    p.noise_alpha = cfg->prior_noise_alpha;
    p.noise_eps = cfg->prior_noise_epsilon;
    p.last_temperature = 1.0f;
    if (cfg->n_temperatures) {
        if (!cfg->temperature_moves || !cfg->temperature_values) throw SpError{CATTUS_B200_EINVAL, "temperature arrays are NULL"};
        for (uint32_t i = 0; i + 1 < cfg->n_temperatures; ++i) {
            if (!(cfg->temperature_values[i] >= 0.0f)) throw SpError{CATTUS_B200_EINVAL, "negative temperature"};
            if (i > 0 && cfg->temperature_moves[i] <= cfg->temperature_moves[i - 1]) throw SpError{CATTUS_B200_EINVAL, "temperature thresholds must be strictly increasing"};
            p.temperatures.emplace_back(cfg->temperature_moves[i], cfg->temperature_values[i]);
        }
        p.last_temperature = cfg->temperature_values[cfg->n_temperatures - 1];
        if (!(p.last_temperature >= 0.0f)) throw SpError{CATTUS_B200_EINVAL, "negative temperature"};
    }
    return p;
}

// Descents per minibatch of cattus_b200_selfplay_run_opts: NULL, 0 or 1 is one leaf in flight.  Minibatches run on the
// device-resident search only.
inline uint32_t selfplay_search_batch(const cattus_b200_selfplay_opts* opts, const cattus_b200_selfplay_cfg& cfg) {
    if (!opts) return 1;
    if (opts->struct_size != sizeof(cattus_b200_selfplay_opts)) throw SpError{CATTUS_B200_EINVAL, "selfplay opts struct_size mismatch"};
    const uint32_t L = opts->search_batch ? opts->search_batch : 1u;
    if (L > 1 && !cfg.device_games)
        throw SpError{CATTUS_B200_EINVAL, "search_batch > 1 needs the device-resident search (device_games > 0); the host-tree driver keeps one leaf in flight"};
    return L;
}

// How a game of the device-resident driver ended (GameRecord::termination; the host driver leaves it 0)
enum Termination : uint8_t { kEndRules = 1, kEndRepetition = 2, kEndMaxMoves = 3 };

struct GameRecord {
    uint32_t game_idx = 0;
    uint8_t winner = 0;
    uint8_t termination = 0;  // Termination
    std::vector<uint16_t> moves;  // hex / ttt: cell index; chess: from | to << 6 | promotion << 12, real board coordinates
    std::vector<std::vector<uint8_t>> entries;
    std::vector<uint8_t> entry_dir;
};

struct Shared {
    // merged from the workers' private counters when they finish (no shared cache line on the per-simulation path)
    uint64_t simulations = 0, searches = 0, evaluations = 0, cache_hits = 0, cache_misses = 0, batches = 0, terminal = 0, speculative = 0;
    uint32_t w1 = 0, w2 = 0, d = 0, games = 0;
    uint64_t minibatches[2] = {0, 0}, collisions[2] = {0, 0};  // device search, per model (1, 2): rounds of descents, collided descents
    std::atomic<uint32_t> next_game{0};
    std::mutex mu;  // records, search_duration, first error
    std::vector<GameRecord> records;
    double search_duration = 0.0;
    double eval_wait = 0.0;
    int error_code = 0;
    std::string error;
    std::atomic<bool> failed{false};
};

// The Dirichlet draw of add_dirichlet_noise (mod.rs:433-439): `count` gamma(alpha) samples; noise[i] / total is the i-th
// component.  Returns the total.
static inline double draw_noise(SplitMix64& rng, float alpha, int count, std::vector<double>& noise) {
    noise.resize(count);
    double tot = 0.0;
    for (int i = 0; i < count; ++i) {
        noise[i] = rng.gamma(static_cast<double>(alpha));
        tot += noise[i];
    }
    return tot;
}

// choose_move_from_probabilities (mod.rs:387-417) over probs in edges() order; returns the index of the chosen entry.
template <class Move>
static int choose_move(const Params& P, size_t history_len, const std::vector<std::pair<Move, float>>& probs, SplitMix64& rng, std::vector<float>& weights) {
    const float temperature = P.temperature_at(history_len / 2);
    int chosen = 0;
    if (temperature == 0.0f) {
        for (size_t i = 1; i < probs.size(); ++i)
            if (!(probs[i].second < probs[chosen].second)) chosen = static_cast<int>(i);  // max_by(total_cmp): last maximum
    } else {
        const float inv = 1.0f / temperature;
        weights.resize(probs.size());
        float tot = 0.0f;
        for (size_t i = 0; i < probs.size(); ++i) {
            weights[i] = static_cast<float>(std::pow(static_cast<double>(probs[i].second), static_cast<double>(inv)));
            tot += weights[i];
        }
        float cum = 0.0f, cum_tot = 0.0f;
        for (size_t i = 0; i < probs.size(); ++i) {
            weights[i] = weights[i] / tot;
            cum_tot += weights[i];
        }
        const double x = rng.next_f64() * static_cast<double>(cum_tot);
        chosen = static_cast<int>(probs.size()) - 1;
        for (size_t i = 0; i < probs.size(); ++i) {
            cum += weights[i];
            if (static_cast<double>(cum) > x) {
                chosen = static_cast<int>(i);
                break;
            }
        }
    }
    return chosen;
}

// write_data_entry + serializers (self_play.rs:248-276, :33-61; serialize/hex.rs:16-28; serialize/ttt.rs:17-22;
// serialize/chess.rs:18-57).  Returns which out_dir (1 or 2) the entry belongs to.
template <class Rules>
static int make_entry(const Rules& R, uint32_t game_idx, const typename Rules::Pos& pos_in,
                      const std::vector<std::pair<typename Rules::Move, float>>& probs_in, uint8_t winner, std::vector<uint8_t>& bytes) {
    using Pos = typename Rules::Pos;
    const int pair_p1[2] = {1, 2}, pair_p2[2] = {2, 1};
    const int dir = (pos_in.turn == 1 ? pair_p1 : pair_p2)[game_idx % 2];
    float w = winner == 0 ? 0.0f : (winner == 1 ? 1.0f : -1.0f);
    if constexpr (Rules::kChess) {
        // ChessSerializer (serialize/chess.rs:18-57).  The stored position and its moves already are the flipped,
        // Player1-to-move view write_data_entry asks for (self_play.rs:260-268); only the winner's sign follows the turn.
        if (pos_in.turn != 1) w = -w;
        std::vector<std::pair<uint16_t, float>> by_idx;
        by_idx.reserve(probs_in.size());
        for (auto& mp : probs_in) by_idx.emplace_back(static_cast<uint16_t>(R.nn_idx(mp.first)), mp.second);
        std::sort(by_idx.begin(), by_idx.end(), [](const auto& a, const auto& b) { return a.first < b.first; });
        if (by_idx.size() > 225) throw SpError{CATTUS_B200_ERANGE, "more than 225 legal moves"};
        uint64_t pl[Rules::kPlanes];
        R.planes(pos_in, pl);
        bytes.assign(Rules::kPlanes * 8 + Rules::kLegalBytes + 225 * 4 + 1, 0);
        uint8_t* p = bytes.data();
        std::memcpy(p, pl, sizeof(pl));
        p += sizeof(pl);
        float probs[225];
        for (float& x : probs) x = -1.0f;
        for (size_t k = 0; k < by_idx.size(); ++k) {
            p[by_idx[k].first >> 3] |= static_cast<uint8_t>(1u << (by_idx[k].first & 7));
            probs[k] = by_idx[k].second;
        }
        p += Rules::kLegalBytes;
        std::memcpy(p, probs, sizeof(probs));
        p += sizeof(probs);
        *p = static_cast<uint8_t>(static_cast<int8_t>(static_cast<int>(w)));
        return dir;
    } else {
        Pos pos = pos_in;
        const bool flipped = pos.turn != 1;
        if (flipped) {
            pos = R.flipped(pos);
            w = -w;
        }
        const int M = R.moves_num();
        std::vector<float> dense(M, -1.0f);
        for (auto& mp : probs_in) dense[flipped ? R.flip_move(mp.first) : mp.first] = mp.second;
        u128 pl[3];
        R.planes(pos, pl);
        const int wpp = R.words_per_plane();
        bytes.resize(3 * wpp * 8 + M * 4 + 1);
        uint8_t* p = bytes.data();
        for (int c = 0; c < 3; ++c)
            for (int k = 0; k < wpp; ++k) {
                const uint64_t word = static_cast<uint64_t>(pl[c] >> (64 * k));
                std::memcpy(p, &word, 8);
                p += 8;
            }
        std::memcpy(p, dense.data(), M * 4);
        p += M * 4;
        *p = static_cast<uint8_t>(static_cast<int8_t>(static_cast<int>(w)));
        return dir;
    }
}

static inline void write_entry_file(const char* dir, uint32_t game_idx, size_t pos_idx, const std::vector<uint8_t>& bytes) {
    char name[64];
    std::snprintf(name, sizeof(name), "/%08u_%03zu.traindata", game_idx, pos_idx);  // format!("{game_idx:#08}_{pos_idx:#03}")
    const std::string path = std::string(dir) + name;
    FILE* f = std::fopen(path.c_str(), "wb");
    if (!f) throw SpError{CATTUS_B200_EINVAL, "cannot create " + path};
    const size_t n = std::fwrite(bytes.data(), 1, bytes.size(), f);
    std::fclose(f);
    if (n != bytes.size()) throw SpError{CATTUS_B200_EINVAL, "short write to " + path};
}

}  // namespace sp
