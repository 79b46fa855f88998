// imx_reset.cuh — episode start: state initialisation, initial observation, and the episode's
// demand trace / noisy-delay mask (replayed from the caller or drawn from Philox), both stored
// period-major so that the step kernel's per-period reads are contiguous across envs.
// Restates reset(): IM_env.py:164-229, MAIM_env.py:176-240, IM_div_env.py:201-302,
// MAIM_div_env.py:240-341.
#pragma once

#include "imx_step.cuh"

namespace imx {

// reset(): inv = init_inv, every other state word 0, and the t = 0 observation.  The initial
// observation is the same m x O block for every env (all history / pipeline slots are 0), so each
// CTA builds that block once in shared memory and the grid then streams it out with coalesced
// 8-byte stores; the zero part of the state is written by the same kernel (no memset nodes).
struct ResetArgs {
    int32_t* zero_base;        // the state block (all fields back to back) ...
    int64_t zero_words;        // ... and its length in int32 words
    int32_t* err;              // [N] watchdog flags, cleared
    const int32_t* demand_in;  // replayed demand trace [N][R][T] of the new episode, or NULL (drawn by demand_generate_kernel)
    int32_t* demand_T;         // [T][R][N]: the trace period-major
    int32_t R, T;
};
constexpr int RESET_T_CHUNK = 8;   // periods one thread transposes

// OT: the observation element type as a template constant (one instantiation per type: no type branches on the fill paths)
template <int DMAX, int PMAX, int OT>
__global__ void __launch_bounds__(256) reset_kernel(const __grid_constant__ StepArgs A_, const __grid_constant__ ResetArgs Z, int div) {
    extern __shared__ __align__(16) double s_tmpl[];                  // [m][O] observation template (8 bytes reserved per element), then int init_inv[m]
    StepArgs A = A_;                                                  // (the fields read below stay parameter-space loads)
    A.obs_type = OT;
    const int m = A.m, O = A.O;
    const int es = obs_elem_bytes(OT);
    int32_t* s_init = reinterpret_cast<int32_t*>(s_tmpl + m * O);
    // everything this kernel writes may still be read by the kernel in front of it (it is launched as a programmatic dependent)
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if ((int)threadIdx.x < m) {
        const int i = threadIdx.x;
        const NodeParams np = load_node(A.nodes + i);
        s_init[i] = np.init_inv;
        if (A.obs) {
            int pipe[DMAX], hd[PMAX], ho[PMAX];
#pragma unroll
            for (int k = 0; k < DMAX; ++k) pipe[k] = 0;
#pragma unroll
            for (int j = 0; j < PMAX; ++j) { hd[j] = 0; ho[j] = 0; }
            write_obs_row<DMAX, PMAX, true>(reinterpret_cast<unsigned char*>(s_tmpl) + (size_t)i * O * es, A, np, i, A.tab ? A.tab + (size_t)i * 4 * A.TL : nullptr, np.init_inv, 0, 0, pipe, hd,
                                      ho, div != 0);
        }
    }
    // (the fills that do not read the template run while the first m threads are still building it: the barrier sits behind them)
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    // zero the whole state block (16 bytes per store), then overwrite inv with init_inv
    int4* z4 = reinterpret_cast<int4*>(Z.zero_base);
    const int64_t n4 = Z.zero_words / 4;
    for (int64_t k = gtid; k < n4; k += stride) z4[k] = make_int4(0, 0, 0, 0);
    for (int64_t k = n4 * 4 + gtid; k < Z.zero_words; k += stride) Z.zero_base[k] = 0;
    for (int64_t k = gtid; k < A.N; k += stride) Z.err[k] = 0;
    if (Z.demand_in) {
        // demand [N][R][T] -> [T][R][N]: one thread per (chunk of RESET_T_CHUNK periods, retailer row, env), env fastest, so the
        // stores of a warp are 32 consecutive words per period and the loads of a thread are one short run of its env's row
        const int R = Z.R, T = Z.T;
        const int chunks = (T + RESET_T_CHUNK - 1) / RESET_T_CHUNK;
        const int64_t rows = A.N * R;
        const int64_t items = rows * chunks;
        for (int64_t k = gtid; k < items; k += stride) {
            const int ch = (int)(k / rows);
            const int64_t idx = k - (int64_t)ch * rows;
            const int r = (int)(idx / A.N);
            const int64_t n = idx - (int64_t)r * A.N;
            const int32_t* src = Z.demand_in + (n * R + r) * T;
            const int t0 = ch * RESET_T_CHUNK;
            int v[RESET_T_CHUNK];
#pragma unroll
            for (int u = 0; u < RESET_T_CHUNK; ++u) v[u] = (t0 + u < T) ? src[t0 + u] : 0;
#pragma unroll
            for (int u = 0; u < RESET_T_CHUNK; ++u)
                if (t0 + u < T) Z.demand_T[((int64_t)(t0 + u) * R + r) * A.N + n] = v[u];
        }
    }
    __syncthreads();                                 // the observation template and init_inv are complete
    if (A.obs) {
        // every env's initial observation is the same m*O-element template: 16-byte stores where the template
        // length allows it, and the position inside the template advances by (stride mod len) per iteration
        // instead of a 64-bit modulo per element
        const int64_t bytes = A.N * m * O * es;
        const int tmpl_bytes = m * O * es;
        if ((tmpl_bytes & 15) == 0 && (reinterpret_cast<uintptr_t>(A.obs) & 15) == 0) {
            const int len = tmpl_bytes / 16;
            const int64_t total = bytes / 16;
            const int4* src = reinterpret_cast<const int4*>(s_tmpl);
            int4* dst = reinterpret_cast<int4*>(A.obs);
            const int step = (int)(stride % len);
            int rem = (int)(gtid % len);
            for (int64_t k = gtid; k < total; k += stride) {
                dst[k] = src[rem];
                rem += step;
                if (rem >= len) rem -= len;
            }
        } else {
            const int len = m * O;
            const int64_t total = A.N * len;
            const int step = (int)(stride % len);
            int rem = (int)(gtid % len);
            for (int64_t k = gtid; k < total; k += stride) {
                if (OT == OBS_BF16) reinterpret_cast<uint16_t*>(A.obs)[k] = reinterpret_cast<const uint16_t*>(s_tmpl)[rem];
                else if (OT == OBS_F32) reinterpret_cast<float*>(A.obs)[k] = reinterpret_cast<const float*>(s_tmpl)[rem];
                else A.obs[k] = s_tmpl[rem];
                rem += step;
                if (rem >= len) rem -= len;
            }
        }
    }
    // inv lives inside the zeroed block: a grid-wide ordering is needed between the zero fill and the
    // init fill of the same words, so the init fill is done by the thread that zeroed the word:
    // inv is the FIRST field of the block (offset 0), words [0, N*m)
    const int64_t cells = A.N * m;
    for (int64_t k = gtid; k < (cells + 3) / 4; k += stride) {
        int rem = (int)((k * 4) % m);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int64_t c = k * 4 + q;
            if (c < cells) A.inv[c] = s_init[rem];
            if (++rem == m) rem = 0;
        }
    }
}

// Philox demand: customer_demand ~ Poisson(mu) / randint(low, high) per (env, retailer, period)
// (scipy.stats .rvs at MAIM_env.py:207,217 — same distributions, different generator).
__global__ void __launch_bounds__(256) demand_generate_kernel(int32_t* __restrict__ out, int64_t N, int R, int T, DemandGen g) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= N * R) return;
    const int r = (int)(idx / N);
    const int64_t n = idx % N;
    for (int t = 0; t < T; t += 2) {
        int d0, d1;
        draw_demand_pair(g, n, r, t, d0, d1);
        out[((int64_t)t * R + r) * N + n] = d0;
        if (t + 1 < T) out[((int64_t)(t + 1) * R + r) * N + n] = d1;
    }
}

// noisy-delay mask [N][T][m] -> [T][N][m]
__global__ void __launch_bounds__(256) mask_transpose_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out,
                                                             int64_t N, int m, int T) {
    const int64_t cell = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= N * m) return;
    const int64_t n = cell / m;
    const int i = (int)(cell % m);
    for (int t = 0; t < T; ++t) out[((int64_t)t * N + n) * m + i] = in[(n * T + t) * m + i];
}

__global__ void __launch_bounds__(256) mask_generate_kernel(uint8_t* __restrict__ out, int64_t N, int m, int T, uint64_t seed,
                                                            int64_t env_offset, uint64_t episode, double thr) {
    const int64_t cell = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= N * m) return;
    const int64_t n = cell / m;
    const int i = (int)(cell % m);
    for (int t = 0; t < T; ++t) out[((int64_t)t * N + n) * m + i] = draw_delay(seed, env_offset + n, i, t, episode, thr) ? 1 : 0;
}

}  // namespace imx
