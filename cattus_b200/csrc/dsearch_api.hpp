// Seam between the self-play C ABI (selfplay.cpp) and the device-resident search (dsearch.cuh, compiled with the engine).
#pragma once

#include "../../include/cattus_b200_selfplay.h"
#include "sp_common.hpp"

namespace cb2 {

// Plays this partition's games with the search trees in HBM (cfg.device_games concurrent games on model1's device);
// records, counters and .traindata files end up in `sh` / the out dirs exactly as the host driver leaves them.
// search_batch: descents per minibatch of model1's and model2's searches (1: one leaf in flight).  Throws sp::SpError.
void dsearch_run(cattus_b200_t* model1, cattus_b200_t* model2, const cattus_b200_selfplay_cfg& cfg, const sp::Params params[2],
                 const uint32_t search_batch[2], sp::Shared& sh);

}  // namespace cb2
