// imx_stats.cuh — small kernels behind the rollout / evaluation entry points: the dfo_func objective and the
// deterministic episode statistics.  Host-TU only (imx_api.cu); not part of the runtime-specialised build.
#pragma once

#include "imx_device.cuh"

namespace imx {

// dfo_func's objective (base_restock_policy.py:41-45): -1 / num_periods * np.sum(prob * rewards) with prob = pmf of the
// episode's demand trace ([T], or [R, T] for a divergent network, where the product broadcasts over the retailer rows) —
// i.e. numpy's pairwise summation over the C-contiguous flattening, element j = prob[j] * rewards[j mod T].  One thread
// per env; numpy's order exactly (loops_utils.h.src, pairwise_sum): sequential below 8 elements, eight running
// accumulators up to 128, above that a recursive split at n/2 rounded down to a multiple of 8.
struct DfoTerm {
    const double* __restrict__ pmf_row;    // [R*T] of this env
    const double* __restrict__ rew;        // step rewards, element t at rew[t * stride]
    int64_t stride;
    int T;
    __device__ __forceinline__ double operator()(int j) const { return __dmul_rn(pmf_row[j], rew[(int64_t)(j % T) * stride]); }
};

// n <= 128: sequential below 8 elements, else eight running accumulators + a sequential tail
__device__ __forceinline__ double np_pairwise_block(const DfoTerm& f, int lo, int n) {
    if (n < 8) {
        double res = 0.0;
        for (int i = 0; i < n; ++i) res = __dadd_rn(res, f(lo + i));
        return res;
    }
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = f(lo + j);
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], f(lo + i + j));
    }
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, f(lo + i));
    return res;
}

// the recursive split above 128 elements, as an explicit post-order walk (n <= 32 * 65535 -> depth <= 16)
__device__ inline double np_pairwise(const DfoTerm& f, int total) {
    struct Frame { int lo, n, stage; double left; };
    Frame st[24];
    int sp = 0;
    double ret = 0.0;
    st[sp].lo = 0; st[sp].n = total; st[sp].stage = 0; st[sp].left = 0.0; ++sp;
    while (sp > 0) {
        const int lo = st[sp - 1].lo, n = st[sp - 1].n, stage = st[sp - 1].stage;
        int n2 = n / 2;
        n2 -= n2 % 8;
        if (stage == 0) {
            if (n <= 128) { ret = np_pairwise_block(f, lo, n); --sp; }
            else { st[sp - 1].stage = 1; st[sp].lo = lo; st[sp].n = n2; st[sp].stage = 0; st[sp].left = 0.0; ++sp; }
        } else if (stage == 1) {
            st[sp - 1].left = ret; st[sp - 1].stage = 2;
            st[sp].lo = lo + n2; st[sp].n = n - n2; st[sp].stage = 0; st[sp].left = 0.0; ++sp;
        } else {
            ret = __dadd_rn(st[sp - 1].left, ret);
            --sp;
        }
    }
    return ret;
}

__global__ void __launch_bounds__(128) dfo_objective_kernel(const double* __restrict__ pmf, const double* __restrict__ step_reward,
                                                            double* __restrict__ dfo, int64_t N, int R, int T) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    DfoTerm f;
    f.pmf_row = pmf + n * (int64_t)R * T;
    f.rew = step_reward + n;
    f.stride = N;
    f.T = T;
    const double s = np_pairwise(f, R * T);
    dfo[n] = __dmul_rn(-1.0 / (double)T, s);              // "-1 / env.num_periods * np.sum(...)": (-1 / T) first, then the product
}

// Episode statistics [n, Σ total, Σ total², then per agent (Σ, Σ²)] in a fixed, deterministic
// order (the payload of the single cross-GPU all-reduce).  Two stages, both of a shape that depends only on N and m:
//   1. stats_slice_kernel: one block per slice of `epb` consecutive envs (stats_envs_per_block: whole warps of envs, up to
//      1024 returns and at most 256 envs per slice), up to four cells per thread.  FUSED: the thread first adds the step
//      rewards of its cells in period order ("reward += r", inv_management.py:223-231; one coalesced row of
//      step_reward [T][cells] per period), writes the episode returns when the caller wants them and leaves them in shared
//      memory — no second pass over the returns; otherwise it loads the returns.  Then one WARP per statistic pair: warp c
//      reduces (Σ, Σ²) of agent c's returns, one more the per-env totals (sum over agents in agent order); lane g adds the
//      envs g, g + 32, ... of the slice in that order and the lanes are added in a fixed shuffle tree.
//   2. stats_final_kernel: one block per statistic adds the slices' partials (strided threads + a fixed tree).
// Both are programmatic dependent launches (griddepcontrol.wait), so their launch latency hides behind the kernel in front.
constexpr int STATS_THREADS = 256;
constexpr int STATS_BLOCKS = 128;                              // slices of the column statistics (imx_eval.cuh)

constexpr int STATS_SLICE_CELLS = 1024;                        // returns one block keeps in shared memory
// envs per slice: as many as fit (whole warps of envs, at most one per thread, at least 32)
static inline int stats_envs_per_block(int cols) {
    int e = (STATS_SLICE_CELLS / cols) & ~31;
    if (e > STATS_THREADS) e = STATS_THREADS;
    return e < 32 ? 32 : e;
}

__device__ __forceinline__ double warp_sum_fixed(double v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v = __dadd_rn(v, __shfl_down_sync(0xffffffffu, v, off));   // (explicit roundings: never contracted)
    return v;
}

template <bool FUSED>
__global__ void __launch_bounds__(STATS_THREADS) stats_slice_kernel(const double* __restrict__ src, double* __restrict__ ret_out,
                                                                    double* __restrict__ partial, int64_t N, int cols, int per_agent, int T,
                                                                    int epb, int nslices) {
    // [epb][stride] returns of the slice; the row stride is odd so that the lanes of phase 2 (one env each) hit distinct banks
    __shared__ double s_ret[STATS_SLICE_CELLS + STATS_THREADS];
    constexpr int MAXK = STATS_SLICE_CELLS / STATS_THREADS;    // cells per thread
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int stride = cols | 1;
    const int64_t env0 = (int64_t)blockIdx.x * epb;
    const int64_t cells = N * cols;
    const int64_t cell0 = env0 * cols;
    const int my_cells = epb * cols;
    asm volatile("griddepcontrol.wait;" ::: "memory");         // (returns at once unless launched as a programmatic dependent)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the final kernel may take its seat; it waits for this grid to complete
    double acc[MAXK];
#pragma unroll
    for (int k = 0; k < MAXK; ++k) {                           // (unrolled: the loads of a thread's cells are all in flight together)
        const int j = tid + k * STATS_THREADS;
        const int64_t c = cell0 + j;
        acc[k] = 0.0;
        if (j < my_cells && c < cells) {
            if (FUSED) {
                int t = 0;
                for (; t + 10 <= T; t += 10) {                 // ten independent loads in flight, added in period order
                    double r[10];
#pragma unroll
                    for (int u = 0; u < 10; ++u) r[u] = src[(int64_t)(t + u) * cells + c];
#pragma unroll
                    for (int u = 0; u < 10; ++u) acc[k] = __dadd_rn(acc[k], r[u]);
                }
                for (; t < T; ++t) acc[k] = __dadd_rn(acc[k], src[(int64_t)t * cells + c]);
                if (ret_out) ret_out[c] = acc[k];
            } else {
                acc[k] = src[c];
            }
        }
    }
#pragma unroll
    for (int k = 0; k < MAXK; ++k) {
        const int j = tid + k * STATS_THREADS;
        if (j < my_cells) s_ret[(j / cols) * stride + (j % cols)] = acc[k];
    }
    __syncthreads();
    // one warp per task: task c < cols = (Σ, Σ²) of agent c's returns, task cols = (Σ, Σ²) of the per-env totals (sum over agents
    // in agent order).  Lane g adds the envs g, g + 32, ... of the slice in that order, then the lanes are added in a fixed tree.
    const int live = (int)(N - env0 < epb ? N - env0 : epb);   // envs of this slice that exist
    for (int task = warp; task <= cols; task += STATS_THREADS / 32) {
        if (task < cols && !per_agent) continue;
        double sum = 0.0, sq = 0.0;
        for (int e = lane; e < live; e += 32) {
            double v;
            if (task < cols) {
                v = s_ret[e * stride + task];
            } else {
                v = 0.0;
                for (int c = 0; c < cols; ++c) v = __dadd_rn(v, s_ret[e * stride + c]);
            }
            sum = __dadd_rn(sum, v);
            sq = __dadd_rn(sq, __dmul_rn(v, v));
        }
        sum = warp_sum_fixed(sum);
        sq = warp_sum_fixed(sq);
        if (lane == 0) {
            const int q = task < cols ? 2 + 2 * task : 0;
            partial[(int64_t)q * nslices + blockIdx.x] = sum;
            partial[(int64_t)(q + 1) * nslices + blockIdx.x] = sq;
        }
    }
}

// One block per statistic: strided threads over the slices' partials, then a fixed shared-memory tree (deterministic).
// accumulate != 0: stats += result (statistics of an evaluation batch build up on the device).
__global__ void __launch_bounds__(STATS_THREADS) stats_final_kernel(const double* __restrict__ partial, double* __restrict__ stats, int64_t N,
                                                                   int nslices, int accumulate) {
    __shared__ double red[STATS_THREADS];
    const int q = blockIdx.x;
    asm volatile("griddepcontrol.wait;" ::: "memory");
    double acc = 0.0;
    for (int b = threadIdx.x; b < nslices; b += STATS_THREADS) acc += partial[(int64_t)q * nslices + b];
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int s = STATS_THREADS / 2; s >= 32; s >>= 1) {
        if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x < 32) {
        const double v = warp_sum_fixed(red[threadIdx.x]);
        if (threadIdx.x == 0) {
            stats[1 + q] = accumulate ? stats[1 + q] + v : v;
            if (q == 0) stats[0] = accumulate ? stats[0] + (double)N : (double)N;
        }
    }
}

// imx_step_eval's composition: one period's rewards into the episode returns in stats_slice_kernel<true>'s order,
// ret[k] = (fresh ? 0.0 : ret[k]) + rew[k] (fresh: period 0, so a reward of -0.0 starts the return at +0.0, as there).
__global__ void __launch_bounds__(256) returns_add_kernel(double* __restrict__ ret, const double* __restrict__ rew, int64_t n, int fresh) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) ret[k] = __dadd_rn(fresh ? 0.0 : ret[k], rew[k]);
}

}  // namespace imx
