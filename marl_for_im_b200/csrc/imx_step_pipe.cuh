// imx_step_pipe.cuh — the step kernel as a persistent, warp-specialised TMA pipeline (runtime-specialised build only).
//
// Why: at the batch sizes an RL loop steps (16 Ki - 128 Ki envs per GPU) the one-tile-per-CTA kernel of
// imx_step_tma.cuh runs as ONE wave whose CTAs all load, then all compute, then all store: launch time =
// fixed floor + issue time + transfer time, added up (profiles/r2_floor_sweep.txt).  Here a CTA stays resident and walks
// over its tiles through a ring of IMX_PIPE_STAGES shared-memory stages:
//   - one PRODUCER thread (an extra warp) issues the bulk loads of tile k + S - 1 while the compute warps work on tile k,
//     waits for a stage's `done` barrier, issues its bulk stores, and refills the stage once the previous stores have
//     been read out of shared memory (cp.async.bulk.wait_group.read 1 — it never waits on the stores it just issued);
//   - the COMPUTE warps wait on the stage's `full` barrier (transaction bytes), run exactly the per-period arithmetic of
//     the other kernels (tile_period, lanes = stages), fence the async proxy and arrive on `done` (one arrival per warp).
// Loads of the next tiles, the arithmetic and the stores of the previous tile overlap inside every SM, and no compute
// warp ever blocks on a store.  Same tile layout, same results bit for bit (tests force both kernels).
// Tiles are assigned statically (blockIdx.x, + gridDim.x, ...).  A dynamic scheduler (one atomicAdd per tile on a word of the
// handle, re-zeroed by the last CTA) was built and measured: 40-60 % SLOWER at every size (config 2 at 65 536 envs: 8.1 us
// against 5.7) — the atomic round trips sit on the producer's critical path and the launch-to-launch differences it was meant to
// remove turned out to be occupancy, not tile-count quantisation (profiles/r2_pipe_sweep.txt, r2_dynamic_scheduler_sweep.txt).
#pragma once

#include "imx_step_tma.cuh"

namespace imx {

struct PipeArgs {
    int32_t n_tiles;           // tiles of E envs this launch covers: envs [0, n_tiles * E)
    int32_t stages;            // ring depth S (2..8); a literal (IMX_PIPE_STAGES) in the specialised build
};

#ifdef IMX_JIT
#ifndef IMX_PIPE_STAGES
#define IMX_PIPE_STAGES 4
#endif
constexpr int PIPE_MAX_STAGES = 8;

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// all but the newest bulk group have been read out of shared memory
__device__ __forceinline__ void bulk_wait_read_but_one() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }

#if defined(IMX_PIPE_MAXNREG)
#define IMX_PIPE_BOUNDS __maxnreg__(IMX_PIPE_MAXNREG)
#else
#define IMX_PIPE_BOUNDS __launch_bounds__(TMA_THREADS + 32)
#endif

template <int M_PAD, int DMAX, int PMAX, int MAXC, bool DIV>
__global__ void IMX_PIPE_BOUNDS step_kernel_pipe(const __grid_constant__ StepArgs A, const __grid_constant__ TileLayout TLY,
                                                 const __grid_constant__ PipeArgs PA IMX_EVAL_PARAM) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t full[PIPE_MAX_STAGES], done[PIPE_MAX_STAGES];
    constexpr int S = IMX_PIPE_STAGES;
    constexpr int CT = TMA_THREADS;                  // compute threads; the producer warp sits behind them
    const int tid = threadIdx.x;
    const int m = KF(m), O = KF(O), E = KT(E);
    const int es = obs_elem_bytes(KF(obs_type));
    const int aes = KF(act_f32) ? 4 : 8;
    const int n_my = (PA.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // tiles blockIdx.x, + gridDim.x, ...
#if IMX_EVAL
    const int32_t stage_bytes = EV.total;            // a stage reserves only the bookkeeping regions this call uses
#else
    constexpr int32_t stage_bytes = KT(total);
#endif

    pdl_launch_dependents();
    if (tid == CT) {
#pragma unroll
        for (int s = 0; s < S; ++s) { mbar_init(&full[s], 1); mbar_init(&done[s], CT / 32); }
        mbar_init_fence();
    }
    __syncthreads();                                 // the only CTA-wide barrier: the roles part ways here

    // ---- what every role that issues bulk loads needs (the producer, and lane 0 of each compute warp for the first ring fill) ----
    const uint32_t b_cell4 = (uint32_t)E * m * 4u, b_cell8 = (uint32_t)E * m * 8u, b_act = (uint32_t)E * m * aes;
    const uint32_t b_pipe = (uint32_t)E * KF(L) * 4u, b_hist = b_cell4 * (uint32_t)KF(P);
    const uint32_t b_bt = (uint32_t)E * KF(NB) * 4u, b_dem = (uint32_t)E * 4u;
    uint32_t b_in = b_act + (uint32_t)KF(R) * b_dem + 3u * b_cell4 + b_pipe;
    if (KF(need_hd)) b_in += b_hist;
    if (KF(need_ho)) b_in += b_hist;
    if (KF(has_carry)) b_in += b_cell4;
    if (DIV && KF(NB) > 0) b_in += b_bt;
#if IMX_EVAL
    const int cols = KF(multi) ? m : 1;
    const uint32_t b_ret = (uint32_t)E * cols * 8u, b_eval = (uint32_t)E * (4 + m) * 8u;
    const bool se_load = A.t > 0;                    // returns / accumulators continue the episode (period 0 starts them at 0.0)
    if (se_load && EV.ret) b_in += b_ret;
    if (se_load && EV.eval) b_in += b_eval;
#endif
    auto first_env = [&](int k) { return ((int64_t)blockIdx.x + (int64_t)k * gridDim.x) * E; };
#if defined(IMX_L2_HINTS) && IMX_L2_HINTS
    const uint64_t pol_stream = l2_policy_evict_first(), pol_keep = l2_policy_evict_last();
#if IMX_L2_HINTS == 2   /* outputs only: the observation stream is evict_first, the rewards evict_last; loads and state untouched */
#define PIPE_LOAD_STREAM(d, s_, b, bar) bulk_load_g2s(d, s_, b, bar)
#define PIPE_LOAD_KEEP(d, s_, b, bar) bulk_load_g2s(d, s_, b, bar)
#define PIPE_STORE_STATE(d, s_, b) bulk_store_only(d, s_, b)
#else
#define PIPE_LOAD_STREAM(d, s_, b, bar) bulk_load_hint(d, s_, b, bar, pol_stream)
#define PIPE_LOAD_KEEP(d, s_, b, bar) bulk_load_hint(d, s_, b, bar, pol_keep)
#define PIPE_STORE_STATE(d, s_, b) bulk_store_hint(d, s_, b, pol_keep)
#endif
#define PIPE_STORE_STREAM(d, s_, b) bulk_store_hint(d, s_, b, pol_stream)
#define PIPE_STORE_KEEP(d, s_, b) bulk_store_hint(d, s_, b, pol_keep)
#else
#define PIPE_STORE_STATE(d, s_, b) bulk_store_only(d, s_, b)
#define PIPE_LOAD_STREAM(d, s_, b, bar) bulk_load_g2s(d, s_, b, bar)
#define PIPE_LOAD_KEEP(d, s_, b, bar) bulk_load_g2s(d, s_, b, bar)
#define PIPE_STORE_STREAM(d, s_, b) bulk_store_only(d, s_, b)
#define PIPE_STORE_KEEP(d, s_, b) bulk_store_only(d, s_, b)
#endif
    // the action tile and demand rows of tile k into L2 while the previous launch drains (see bulk_prefetch_l2)
    auto prefetch_inputs = [&](int k) {
#if !defined(IMX_NO_ACT_PREFETCH)
        bulk_prefetch_l2(reinterpret_cast<const unsigned char*>(A.actions) + first_env(k) * m * aes, b_act);
        for (int r = 0; r < KF(R); ++r)              // (the demand trace was written at reset() and is long evicted)
            bulk_prefetch_l2(A.demand_T + ((int64_t)A.t * KF(R) + r) * A.N + first_env(k), b_dem);
#endif
    };
    auto issue_loads = [&](int k) {
        const int s = k % S;
        unsigned char* st = smem + (size_t)s * stage_bytes;
        const int64_t n0 = first_env(k);
        uint64_t* bar = &full[s];
        mbar_expect_tx(bar, b_in);
        PIPE_LOAD_STREAM(st + KT(off_act), reinterpret_cast<const unsigned char*>(A.actions) + n0 * m * aes, b_act, bar);
        for (int r = 0; r < KF(R); ++r)
            PIPE_LOAD_STREAM(st + KT(off_dem) + (size_t)r * b_dem, A.demand_T + ((int64_t)A.t * KF(R) + r) * A.N + n0, b_dem, bar);
        PIPE_LOAD_KEEP(st + KT(off_inv), A.inv + n0 * m, b_cell4, bar);
        PIPE_LOAD_KEEP(st + KT(off_bl), A.backlog + n0 * m, b_cell4, bar);
        PIPE_LOAD_KEEP(st + KT(off_ou), A.order_u + n0 * m, b_cell4, bar);
        PIPE_LOAD_KEEP(st + KT(off_pipe), A.pipe + n0 * KF(L), b_pipe, bar);
        if (KF(need_hd)) PIPE_LOAD_KEEP(st + KT(off_hd), A.hist_d + n0 * m * KF(P), b_hist, bar);
        if (KF(need_ho)) PIPE_LOAD_KEEP(st + KT(off_ho), A.hist_o + n0 * m * KF(P), b_hist, bar);
        if (KF(has_carry)) PIPE_LOAD_KEEP(st + KT(off_carry), A.carry + n0 * m, b_cell4, bar);
        if (DIV && KF(NB) > 0) PIPE_LOAD_KEEP(st + KT(off_bt), A.bt + n0 * KF(NB), b_bt, bar);
#if IMX_EVAL
        if (se_load && EV.ret) PIPE_LOAD_KEEP(st + EV.off_ret, EV.ret + n0 * cols, b_ret, bar);
        if (se_load && EV.eval) PIPE_LOAD_KEEP(st + EV.off_eval, EV.eval + n0 * (4 + m), b_eval, bar);
#endif
    };

    // The first ring fill is the launch's critical path: one thread issuing S tiles x 7-10 bulk loads one after the other
    // puts the last tile's loads ~0.5 us behind the first's (each bulk copy is ~10 dependent uniform-datapath instructions).
    // The compute warps have nothing to do until their first tile lands, so the fill is dealt round-robin over ALL warps:
    // tile k of the fill is issued by warp k mod NW (0 = producer warp, w + 1 = compute warp w).
    constexpr int NW = 1 + CT / 32;
    const int pre = n_my < S ? n_my : S;
    if (tid >= CT) {
        if (tid != CT) return;
        // ---------------------------------------------------------------- producer ---------------------------------
        auto issue_stores = [&](int k) {
            const int s = k % S;
            const unsigned char* st = smem + (size_t)s * stage_bytes;
            const int64_t n0 = first_env(k);
            if (KHAS(cc)) PIPE_STORE_STREAM(reinterpret_cast<unsigned char*>(A.cc) + n0 * m * A.cc_W * es, st + KT(off_cc), (uint32_t)E * m * A.cc_W * es);
            if (KHAS(obs)) PIPE_STORE_STREAM(reinterpret_cast<unsigned char*>(A.obs) + n0 * m * O * es, st + KT(off_obs), (uint32_t)E * m * O * es);
            if (!IMX_EVAL || A.reward) PIPE_STORE_KEEP(A.reward + (KF(multi) ? n0 * m : n0), st + KT(off_rew), KF(multi) ? b_cell8 : (uint32_t)E * 8u);
            PIPE_STORE_STATE(A.inv + n0 * m, st + KT(off_inv), b_cell4);
            PIPE_STORE_STATE(A.backlog + n0 * m, st + KT(off_bl), b_cell4);
            PIPE_STORE_STATE(A.order_u + n0 * m, st + KT(off_ou), b_cell4);
            PIPE_STORE_STATE(A.pipe + n0 * KF(L), st + KT(off_pipe), b_pipe);
            if (KF(need_hd)) PIPE_STORE_STATE(A.hist_d + n0 * m * KF(P), st + KT(off_hd), b_hist);
            if (KF(need_ho)) PIPE_STORE_STATE(A.hist_o + n0 * m * KF(P), st + KT(off_ho), b_hist);
            if (KF(has_carry)) PIPE_STORE_STATE(A.carry + n0 * m, st + KT(off_carry), b_cell4);
            if (DIV && KF(NB) > 0) PIPE_STORE_STATE(A.bt + n0 * KF(NB), st + KT(off_bt), b_bt);
#if IMX_EVAL
            // returns and accumulators travel like state, the diagnostics like the observation stream (one commit group per tile)
            if (EV.ret) PIPE_STORE_STATE(EV.ret + n0 * cols, st + EV.off_ret, b_ret);
            if (EV.eval) PIPE_STORE_STATE(EV.eval + n0 * (4 + m), st + EV.off_eval, b_eval);
            if (EV.info.demand_dev) PIPE_STORE_STREAM(EV.info.demand_dev + n0 * m, st + EV.off_idem, b_cell4);
            if (EV.info.ship_dev) PIPE_STORE_STREAM(EV.info.ship_dev + n0 * m, st + EV.off_iship, b_cell4);
            if (EV.info.acquisition_dev) PIPE_STORE_STREAM(EV.info.acquisition_dev + n0 * m, st + EV.off_iacq, b_cell4);
            if (EV.info.order_dev) PIPE_STORE_STREAM(EV.info.order_dev + n0 * m, st + EV.off_iord, b_cell4);
            if (EV.info.profit_dev) PIPE_STORE_STREAM(EV.info.profit_dev + n0 * m, st + EV.off_prof, b_cell8);
#endif
            bulk_commit();
        };
        for (int k = 0; k < pre; k += NW) prefetch_inputs(k);
        pdl_wait();                                  // state written by the previous step must be complete and visible
        for (int k = 0; k < pre; k += NW) issue_loads(k);
        for (int k = 0; k < n_my; ++k) {
            mbar_wait(&done[k % S], (uint32_t)((k / S) & 1));
            issue_stores(k);
            if (S >= 3) {
                // refill the stage tile k - 1 lived in: its stores were issued one tile ago and are (nearly always) read out
                if (k >= 1 && k - 1 + S < n_my) { bulk_wait_read_but_one(); issue_loads(k - 1 + S); }
            } else {
                if (k + S < n_my) { bulk_wait_read_all(); issue_loads(k + S); }
            }
        }
        bulk_wait_read_all();                        // shared memory must outlive the bulk engine's reads
        return;
    }

    // -------------------------------------------------------------------- compute warps ------------------------------
    const LaneCtx<MAXC> L = make_lane_ctx<M_PAD, MAXC, DIV>(A, tid);
    if ((tid & 31) == 0 && (tid >> 5) + 1 < pre) {   // this warp's share of the first ring fill (tiles w + 1, w + 1 + NW, ...)
        for (int k = (tid >> 5) + 1; k < pre; k += NW) prefetch_inputs(k);
        pdl_wait();
        for (int k = (tid >> 5) + 1; k < pre; k += NW) issue_loads(k);
    }
    // (prefetching the rescale table into L1 here was measured: 5.5 -> 8.3 us per launch at 65 536 envs, profiles/r2_act_prefetch_ab.txt)
    for (int k = 0; k < n_my; ++k) {
        const int s = k % S;
        unsigned char* st = smem + (size_t)s * stage_bytes;
        const TileSmem T = {st + KT(off_act), reinterpret_cast<const int32_t*>(st + KT(off_dem)),
                            reinterpret_cast<int32_t*>(st + KT(off_inv)), reinterpret_cast<int32_t*>(st + KT(off_bl)),
                            reinterpret_cast<int32_t*>(st + KT(off_ou)), reinterpret_cast<int32_t*>(st + KT(off_pipe)),
                            reinterpret_cast<int32_t*>(st + KT(off_hd)), reinterpret_cast<int32_t*>(st + KT(off_ho)),
                            reinterpret_cast<int32_t*>(st + KT(off_carry)), reinterpret_cast<int32_t*>(st + KT(off_bt)),
                            st + KT(off_obs), reinterpret_cast<double*>(st + KT(off_rew))
#if IMX_EVAL
                            , (EV.eval || EV.info.profit_dev) ? reinterpret_cast<double*>(st + EV.off_prof) : nullptr,
                            EV.ret ? reinterpret_cast<double*>(st + EV.off_ret) : nullptr,
                            EV.info.demand_dev ? reinterpret_cast<int32_t*>(st + EV.off_idem) : nullptr,
                            EV.info.ship_dev ? reinterpret_cast<int32_t*>(st + EV.off_iship) : nullptr,
                            EV.info.acquisition_dev ? reinterpret_cast<int32_t*>(st + EV.off_iacq) : nullptr,
                            EV.info.order_dev ? reinterpret_cast<int32_t*>(st + EV.off_iord) : nullptr
#endif
                            };
        const int64_t n0 = ((int64_t)blockIdx.x + (int64_t)k * gridDim.x) * E;
        mbar_wait(&full[s], (uint32_t)((k / S) & 1));
#if IMX_USE_STEP_ET
        tile_period_et<IMX_K_m, DMAX, PMAX, MAXC, DIV, false, (bool)IMX_EVAL>(A, TLY, T, tid, A.t, n0, []() {});
#if IMX_EVAL
        if (EV.eval) step_eval_env_pass(A, TLY, EV, st, tid);           // this thread simulated env tid
#endif
#else
        // replayed / Philox noisy-delay outcome of this lane's (env, stage) for this period (written by reset(), long complete)
        const bool delayed = (KF(noisy) && L.ok) ? (A.mask_T[((int64_t)A.t * A.N + n0 + L.e_loc) * m + L.i] != 0) : false;
        tile_period<M_PAD, DMAX, PMAX, MAXC, DIV, false, false, (bool)IMX_EVAL>(A, TLY, T, L, A.t, 0, n0, delayed, []() {});
#if IMX_EVAL
        if (EV.eval) {                               // the env's cells sit in this warp: no barrier across compute warps
            __syncwarp();
            if (L.ok && L.i == 0) step_eval_env_pass(A, TLY, EV, st, L.e_loc);
        }
#endif
#endif
        if (KHAS(cc)) cc_build<MAXC>(A, TLY, T, st, L, CT);
        fence_proxy_async_smem();                    // this thread's tile writes, before the bulk engine reads them
        __syncwarp();
        if (L.lane == 0) mbar_arrive(&done[s]);      // release: the producer's wait acquires the whole warp's writes
    }
}
#endif  // IMX_JIT

}  // namespace imx
