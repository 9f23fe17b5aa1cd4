// Host-side dispatch of the lane-split rollout kernel for one segment count N (see lane_rollout.cuh).
// Each lane_nK.cu translation unit instantiates launch_lane_rollout_n<K>.
#pragma once
#include "lane2_rollout.cuh"
#include "launch.cuh"

namespace swm {

// lanes per environment of the lane-split kernel for an n-segment swimmer (LaneSplit<N>::L)
inline int lane_split_lanes(int n) { return (n + 1 <= 4) ? 4 : (n + 1 <= 8) ? 8 : 16; }

// what the lane-split kernels implement: gym dynamics, fixed actions or linear policies (V1 / V2, with or
// without moments), no action clipping; per-step screening only in the warp-specialised kernels (f_warps >= 1) and
// only for plain linear policies
inline bool lane_split_supported(const RolloutArgs& a, const RolloutFlags& f, int f_warps = 0) {
  if (f.variant != SWM_DYN_GYM || a.clip) return false;
  if (f.screen) return f_warps >= 1 && f.linear && !f.norm && !f.stats;
  if (!f.linear) return !f.norm && !f.stats;
  return !(f.stats && !f.norm);
}

// f_warps: 0 = one warp per lane group (lane_rollout.cuh); 1 / 2 = the warp-specialised form with that many
// operator warps beside the main warp (lane2_rollout.cuh)
template <int N> int launch_lane_rollout_n(const RolloutArgs& a, const RolloutFlags& f, int f_warps, cudaStream_t st);
// model-set mode (see launch_rollout_models_n): linear policies, V1 / V2 without statistics, no screening
template <int N> int launch_lane_rollout_models_n(const RolloutArgs& a, const SimModels& models, const RolloutFlags& f,
                                                  int f_warps, cudaStream_t st);

#ifdef SWM_INSTANTIATE_LANE_N

// One launch of the lane-split kernel of f_warps (the warp-specialised form whenever SCREEN) with the second kernel
// argument `second` (the models of the model-set mode, else empty) and grid_y CTA rows.
template <int N, bool LINEAR, bool NORM, bool STATS, bool SCREEN, bool MODELS, typename Second>
static int launch_lane(const RolloutArgs& a, const Second& second, unsigned grid_y, int f_warps, cudaStream_t st) {
  constexpr int G = LaneSplit<N>::G;
  const long long blocks = (a.B + G - 1) / G;
  if (blocks > 0x7fffffffLL) return SWM_ERR_BAD_ARG;
  const dim3 grid((unsigned)blocks, grid_y);
  if (f_warps == 2) lane2_rollout_kernel<N, LINEAR, NORM, STATS, 2, SCREEN, MODELS><<<grid, 96, 0, st>>>(a, second);
  else if (f_warps == 1 || SCREEN) lane2_rollout_kernel<N, LINEAR, NORM, STATS, 1, SCREEN, MODELS><<<grid, 64, 0, st>>>(a, second);
  else lane_rollout_kernel<N, LINEAR, NORM, STATS, MODELS><<<grid, kLaneBlock, 0, st>>>(a, second);
  return cudaPeekAtLastError() == cudaSuccess ? SWM_OK : SWM_ERR_CUDA;
}

template <int N>
int launch_lane_rollout_n(const RolloutArgs& a, const RolloutFlags& f, int f_warps, cudaStream_t st) {
  if (!lane_split_supported(a, f, f_warps)) return SWM_ERR_UNSUPPORTED;
  const NoCostForms none;
  if (f.screen) return launch_lane<N, true, false, false, true, false>(a, none, 1, f_warps, st);
  if (!f.linear) return launch_lane<N, false, false, false, false, false>(a, none, 1, f_warps, st);
  if (f.norm && f.stats) return launch_lane<N, true, true, true, false, false>(a, none, 1, f_warps, st);
  if (f.norm) return launch_lane<N, true, true, false, false, false>(a, none, 1, f_warps, st);
  return launch_lane<N, true, false, false, false, false>(a, none, 1, f_warps, st);
}

template <int N>
int launch_lane_rollout_models_n(const RolloutArgs& a, const SimModels& models, const RolloutFlags& f, int f_warps,
                                 cudaStream_t st) {
  if (!lane_split_supported(a, f, f_warps) || !f.linear || f.screen || f.stats) return SWM_ERR_UNSUPPORTED;
  if (f.norm) return launch_lane<N, true, true, false, false, true>(a, models, models.M, f_warps, st);
  return launch_lane<N, true, false, false, false, true>(a, models, models.M, f_warps, st);
}

template int launch_lane_rollout_n<SWM_INSTANTIATE_LANE_N>(const RolloutArgs&, const RolloutFlags&, int, cudaStream_t);
template int launch_lane_rollout_models_n<SWM_INSTANTIATE_LANE_N>(const RolloutArgs&, const SimModels&,
                                                                  const RolloutFlags&, int, cudaStream_t);

#endif  // SWM_INSTANTIATE_LANE_N

}  // namespace swm
