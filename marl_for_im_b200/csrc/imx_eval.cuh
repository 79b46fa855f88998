// imx_eval.cuh — per-episode accumulators of the reference's evaluation loops, kept on the device.
//
// MA_inv_management.py:538-587 (same loop in CC_inv_management.py:512-556, CC_inv_management_div.py:500-544,
// MA_inv_management_div.py, inv_management.py:573-606 and the LP replay loops, e.g. DSHLP_4.py:896-928):
//
//     for every step:   for m in stages:   episode_reward    += reward[agent m]
//                                          stage_rewards[m]  += info[agent m]['profit']
//                                          total_step_inv    += rev_scale(obs[m][0], 0, inv_max[m], a, b)
//                                          total_step_bl     += rev_scale(obs[m][1], 0, inv_max[m], a, b)
//                       total_inventory  += total_step_inv ;  total_backlog += total_step_bl
//                       customer_backlog += rev_scale(obs[0][1], 0, inv_max[0], a, b)
//
// The LP loops read a non-standardised env, so their `sum(s[:, 0])` is the same sum without rev_scale.
// One thread per env performs exactly these float64 operations in this order, so the accumulators are
// bit-identical to the host loop.  Row layout of acc [N][4 + m]:
//     {episode_reward, total_inventory, total_backlog, customer_backlog, stage_profit[0..m-1]}
#pragma once
#include "imx_device.cuh"

namespace imx {

constexpr int EVAL_FIXED = 4;

struct EvalArgs {
    const void* __restrict__ obs;        // [N][m][O] in the handle's observation type (OBS_F64 / OBS_F32 / OBS_BF16)
    const double* __restrict__ reward;   // MAIM kinds [N][m], IM kinds [N]
    const double* __restrict__ profit;   // [N][m] or null (stage_profit columns are then left untouched)
    double* __restrict__ acc;            // [N][4 + m]
    const NodeParams* __restrict__ nodes;
    int64_t N;
    int32_t m, O, multi, obs_type;
    int32_t rescaled;                    // observations are standardised: undo with rev_scale (MAIM_env.py:509-519)
    int32_t reset;                       // start a new episode: accumulators begin at 0 instead of acc's contents
    double a, bma;
};

__global__ void __launch_bounds__(256) eval_accumulate_kernel(const __grid_constant__ EvalArgs E) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= E.N) return;
    const int m = E.m, O = E.O, W = EVAL_FIXED + m;
    double* row = E.acc + n * W;
    double ep = E.reset ? 0.0 : row[0];
    double step_inv = 0.0, step_bl = 0.0, cust = 0.0;
    if (!E.multi) ep = __dadd_rn(ep, E.reward[n]);                      // inv_management.py:596 "episode_reward += reward"
    for (int i = 0; i < m; ++i) {
        double x0, x1;
        if (E.obs_type == OBS_BF16) {
            const uint16_t* o = reinterpret_cast<const uint16_t*>(E.obs) + (n * m + i) * O;
            x0 = (double)bf16_to_f32(o[0]); x1 = (double)bf16_to_f32(o[1]);
        } else if (E.obs_type == OBS_F32) {
            const float* o = reinterpret_cast<const float*>(E.obs) + (n * m + i) * O;
            x0 = (double)o[0]; x1 = (double)o[1];
        } else {
            const double* o = reinterpret_cast<const double*>(E.obs) + (n * m + i) * O;
            x0 = o[0]; x1 = o[1];
        }
        if (E.rescaled) {
            const double vmax = (double)E.nodes[i].inv_max;             // the loops use inv_max[m] for BOTH fields
            x0 = rev_scale_dev(x0, vmax, E.a, E.bma);
            x1 = rev_scale_dev(x1, vmax, E.a, E.bma);
        }
        if (E.multi) ep = __dadd_rn(ep, E.reward[n * m + i]);
        if (E.profit) row[EVAL_FIXED + i] = __dadd_rn(E.reset ? 0.0 : row[EVAL_FIXED + i], E.profit[n * m + i]);
        else if (E.reset) row[EVAL_FIXED + i] = 0.0;
        step_inv = __dadd_rn(step_inv, x0);
        step_bl = __dadd_rn(step_bl, x1);
        if (i == 0) cust = x1;
    }
    row[0] = ep;
    row[1] = __dadd_rn(E.reset ? 0.0 : row[1], step_inv);
    row[2] = __dadd_rn(E.reset ? 0.0 : row[2], step_bl);
    row[3] = __dadd_rn(E.reset ? 0.0 : row[3], cust);
}

// Column statistics of a [N][W] float64 matrix: stats = {n, then per column (Σ, Σ²)} — what
// np.mean / np.std over the episode lists need (MA_inv_management.py:589-600).  Same fixed-shape
// two-stage reduction as the return statistics: the result depends only on N.
__global__ void __launch_bounds__(STATS_THREADS) column_stats_partial_kernel(const double* __restrict__ mat, double* __restrict__ partial,
                                                                             int64_t N, int W) {
    __shared__ double red[STATS_THREADS];
    const int q = blockIdx.y;                       // statistic: column q/2, square if odd
    const int col = q >> 1;
    const int64_t per_block = (N + STATS_BLOCKS - 1) / STATS_BLOCKS;
    const int64_t lo = (int64_t)blockIdx.x * per_block;
    const int64_t hi = lo + per_block < N ? lo + per_block : N;
    double acc = 0.0;
    for (int64_t n = lo + threadIdx.x; n < hi; n += STATS_THREADS) {
        const double v = mat[n * W + col];
        acc += (q & 1) ? v * v : v;
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int s = STATS_THREADS / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[q * STATS_BLOCKS + blockIdx.x] = red[0];
}

}  // namespace imx
