// imx_cc.cuh — centralised-critic observation build (SURVEY §8(f) rank 1).
// Restates central_critic_observer (models/CC_Model.py:196-214) + the opponent-action fill of
// FillInActions (:165-193) / the hand-built CC obs of the evaluation loops
// (CC_inv_management.py:516-528) for a whole batch: for every agent i of every env the flat vector
//     [ opponent_action (m-1) | opponent_obs (m-1)*O | own_obs O ]
// (RLlib flattens the dict in sorted key order), opponents in agent order skipping i, opponent
// actions clipped to [lo, hi] (zeros when no action tensor is given, as the observer does at
// sampling time).  Pure gather, HBM-bound: one thread per output element, coalesced writes.
#pragma once

#include "imx_device.cuh"

namespace imx {

// Element types: double, float, and Bf16 (bit pattern; widened exactly, narrowed as torch does: float64 -> float32 -> bfloat16).
struct Bf16 { uint16_t u; };
__device__ __forceinline__ double widen(double x) { return x; }
__device__ __forceinline__ double widen(float x) { return (double)x; }
__device__ __forceinline__ double widen(Bf16 x) { return (double)bf16_to_f32(x.u); }
template <typename T> __device__ __forceinline__ T narrow(double v);
template <> __device__ __forceinline__ double narrow<double>(double v) { return v; }
template <> __device__ __forceinline__ float narrow<float>(double v) { return (float)v; }
template <> __device__ __forceinline__ Bf16 narrow<Bf16>(double v) { return Bf16{f32_to_bf16((float)v)}; }

template <typename InT, typename OutT>
__global__ void __launch_bounds__(256) cc_observer_kernel(const InT* __restrict__ obs, const void* __restrict__ actions, int act_f32,
                                                          OutT* __restrict__ out, int64_t N, int m, int O, double lo, double hi) {
    const int W = (m - 1) * (1 + O) + O;
    const int64_t total = N * m * W;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
        const int64_t n = idx / ((int64_t)m * W);
        const int rem = (int)(idx - n * m * W);
        const int i = rem / W, w = rem - i * W;
        double v;
        if (w < m - 1) {
            const int j = w < i ? w : w + 1;
            v = actions ? clip_np(load_action(actions, n * m + j, act_f32 != 0), lo, hi) : 0.0;
        } else if (w < (m - 1) * (1 + O)) {
            const int q = w - (m - 1);
            const int slot = q / O, k = q - slot * O;
            const int j = slot < i ? slot : slot + 1;
            v = widen(obs[(n * m + j) * O + k]);
        } else {
            v = widen(obs[(n * m + i) * O + (w - (m - 1) * (1 + O))]);
        }
        out[idx] = narrow<OutT>(v);
    }
}

}  // namespace imx
