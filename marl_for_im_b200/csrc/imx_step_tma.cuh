// imx_step_tma.cuh — the step kernel with TMA-staged tiles (the fast path).
//
// One CTA = one tile of E = 256 / M_PAD consecutive environments.  Because state and I/O are
// structure-of-arrays with the env index slowest, every field of a tile is ONE contiguous byte
// range in HBM:  actions E*m*8 (float32: E*m*4),  inv / backlog / order_u E*m*4 each,  pipe E*L*4,  hist E*m*P*4,
// demand E*4 per retailer row,  obs E*m*O*8,  reward E*m*8.
//   1. one elected thread arms an mbarrier with the tile's byte count and issues one
//      cp.async.bulk (global -> shared, SASS UBLKCP) per field;
//   2. all lanes wait on the mbarrier, then work out of shared memory with per-thread constant
//      offsets (lanes = stages, shuffles for the stage coupling — same arithmetic as
//      imx_step.cuh, shared through the same device functions);
//   3. the new state is written in place in shared memory, observations and rewards into their
//      tiles; every thread fences the async proxy, the CTA syncs, and the elected thread issues
//      one bulk store (shared -> global) per field.
// The per-lane instruction stream therefore contains no global address arithmetic at all, which is
// what bounds the direct kernel (see profiles/).  Tail tiles (N % E != 0), unaligned caller
// buffers and the replayed noisy-delay mask go through the direct kernel in imx_step.cuh.
#pragma once

#include "imx_step.cuh"

namespace imx {

// Threads per CTA of the TMA kernel = M_PAD * (envs per tile).  512 for the ahead-of-time build (an
// upper bound: the host launches 128 or 256); the runtime-specialised build pins the value it launches with.
#ifndef IMX_TMA_THREADS
#define IMX_TMA_THREADS 512
#endif
constexpr int TMA_THREADS = IMX_TMA_THREADS;

// Byte offsets of the tile regions inside dynamic shared memory (all multiples of 128).
struct TileLayout {
    int32_t E;                 // envs per tile
    int32_t off_act, off_inv, off_bl, off_ou, off_pipe, off_hd, off_ho, off_carry, off_bt, off_dem, off_obs, off_rew;
    int32_t total;             // dynamic shared memory bytes
    // second buffers of the per-period inputs (actions, demand), used by multi-period launches
    int32_t off_act2, off_dem2;
    int32_t total2;            // dynamic shared memory bytes of a multi-period launch (second buffers sit behind `total`)
    int32_t off_cc;            // centralised-critic rows [E][m][W] (layouts built for imx_step_cc only; inside `total`)
};

// One whole stored-plan episode per launch (imx_replay_episode, step_kernel_tma_episode): what the kernel needs beyond the
// multi-period StepArgs.  The episode regions of shared memory sit behind TileLayout.total2 (the per-period demand rows of
// that layout are unused: the episode's whole trace is resident instead).
struct EpisodeArgs {
    const int32_t* __restrict__ demand;   // replayed trace [N][R][T] read in place (one bulk copy per tile), or null: Philox draws
    const uint8_t* __restrict__ mask;     // replayed noisy-delay outcomes [N][T][m], or null: Philox draws (when A.noisy)
    double* __restrict__ ret;             // episode returns [N][m] / [N], or null
    double* __restrict__ eval;            // evaluation-loop accumulators [N][4 + m], or null
    DemandGen gen;                        // the Philox stream imx_reset would draw this episode from
    double delay_thr;                     // noisy_delay_threshold of the Philox delay draws
    int32_t off_edem;                     // [E][R][T] int32 demand of the tile's envs
    int32_t off_ret;                      // [E][m] / [E] float64 returns
    int32_t off_eval;                     // [E][4 + m] float64 accumulators
    int32_t off_prof;                     // [E][m] float64 profits of the current period (eval only)
    int32_t total;                        // dynamic shared memory bytes
    int32_t rescaled;                     // the state is standardised: the accumulators undo the scaling (rev_scale)
};

// Noisy-delay outcome of (local env n, node i, period t) in an episode launch: the replayed mask, or the draw
// mask_generate_kernel makes for imx_reset(noisy = 1) of the same episode.
__device__ __forceinline__ bool episode_delayed(const EpisodeArgs& EA, int64_t n, int m, int T, int i, int t) {
    if (EA.mask) return EA.mask[(n * T + t) * m + i] != 0;
    return draw_delay(EA.gen.seed, EA.gen.env_offset + n, i, t, EA.gen.episode, EA.delay_thr);
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load_g2s(void* sdst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sdst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done = 0;
    for (int spin = 0; !done; ++spin) {
        // the suspend-time hint lets the warp sleep in hardware until the transaction completes instead of
        // re-issuing the probe (the spin was 11 % of the divergent kernel's issue slots)
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n selp.b32 %0, 1, 0, p;\n}"
                     : "=r"(done)
                     : "r"(smem_u32(bar)), "r"(parity), "r"(0x989680u)
                     : "memory");
        if (spin > (1 << 24)) __trap();      // a lost transaction must fail loudly, not hang the GPU
    }
}
__device__ __forceinline__ void bulk_store_only(void* gdst, const void* ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// L2 eviction priorities for the bulk copies (runtime-specialised build, IMX_L2_HINTS): the observation / critic-row stream is
// written once and never read by the path (evict_first), the state is read and rewritten every period and the step rewards are
// read back by the episode statistics (evict_last) — so the write-once stream does not push the re-used lines out of L2.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void bulk_store_hint(void* gdst, const void* ssrc, uint32_t bytes, uint64_t policy) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(gdst), "r"(smem_u32(ssrc)),
                 "r"(bytes), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ void bulk_load_hint(void* sdst, const void* gsrc, uint32_t bytes, uint64_t* bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                     smem_u32(sdst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
                 : "memory");
}
// L2 prefetch of a global byte range (a hint: it moves no data into the SM and cannot observe a stale value — L2 is the
// point of coherence, a later write by the kernel in front simply updates the line).  Issued BEFORE griddepcontrol.wait for
// the one input a step reads that is cold: the caller's action block (in the benchmark loop it comes from HBM every period,
// while the state was written into L2 by the previous step), so its DRAM latency overlaps the previous launch's drain.
__device__ __forceinline__ void bulk_prefetch_l2(const void* gsrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gsrc), "r"(bytes) : "memory");
}

// Programmatic dependent launch (sm_90+): back-to-back step() launches are chained with
// cudaLaunchAttributeProgrammaticStreamSerialization, so the next grid may start its prologue
// (barrier init, per-lane constants) while this one drains; it blocks in pdl_wait() until the
// previous grid has completed and its writes are visible, before touching any state.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Shared-memory bank conflicts of the observation tile.  A lane writes its agent's row (O elements) into the tile, whose
// layout must equal the global [E][m][O] block (it leaves as one linear bulk copy), so consecutive lanes are one row apart.
// When the row is c = O * es / 16 chunks of 16 bytes and g = gcd(c, 8) > 1, the lanes of a quarter-warp that are 8 / g
// apart hit the same banks with the same chunk (O = 8 float64: 64-byte rows, 4-way conflict, 16 wavefronts per STS.128
// instead of 4 — 60 % of all shared-memory wavefronts of the 8-stage kernel, profiles/r1_ncu_step_kernel_8stage_1Mi_envs.txt).
// Cure: every lane stores the SAME chunks in a ROTATED order — at store q lane l writes chunk (q + r) mod c with
// r = (l mod 8) / (8 / g) — which makes the eight lanes of a quarter-warp cover eight different 16-byte bank groups.
// The rotation is a barrel of selects on registers (static indices only).  Runtime-specialised build only (O is a literal).
#ifdef IMX_JIT
#define IMX_K_OBS_ES (IMX_K_obs_type == 2 ? 2 : IMX_K_obs_type == 1 ? 4 : 8)   // = obs_elem_bytes(IMX_K_obs_type), for #if
#endif
#if defined(IMX_JIT) && ((IMX_K_O * IMX_K_OBS_ES) % 32 == 0) && ((IMX_K_O * IMX_K_OBS_ES) <= 256)
#define IMX_OBS_ROTATE 1          // the row is an even number (<= 16) of 16-byte chunks: gcd(c, 8) > 1
#endif
#ifdef IMX_OBS_ROTATE
__host__ __device__ constexpr int obs_gcd8(int c) { return (c % 8 == 0) ? 8 : (c % 4 == 0) ? 4 : (c % 2 == 0) ? 2 : 1; }
constexpr int OBS_ROW_BYTES = IMX_K_O * IMX_K_OBS_ES;
constexpr int OBS_ROW_CHUNKS = OBS_ROW_BYTES / 16;
constexpr int OBS_ROT_G = obs_gcd8(OBS_ROW_CHUNKS);

struct ObsChunk { unsigned long long lo, hi; };
__device__ __forceinline__ ObsChunk obs_sel(bool c, const ObsChunk& a, const ObsChunk& b) { ObsChunk r; r.lo = c ? a.lo : b.lo; r.hi = c ? a.hi : b.hi; return r; }

__device__ __forceinline__ void store_row_rotated(unsigned char* dst, const unsigned long long (&w)[OBS_ROW_BYTES / 8], int lane) {
    constexpr int C = OBS_ROW_CHUNKS, G = OBS_ROT_G;
    const int r = (lane & 7) / (8 / G);                 // 0 .. G-1
    ObsChunk cur[C], nxt[C];
#pragma unroll
    for (int q = 0; q < C; ++q) { cur[q].lo = w[2 * q]; cur[q].hi = w[2 * q + 1]; }
#pragma unroll
    for (int bit = 1; bit < G; bit <<= 1) {             // cur[q] <- chunk (q + r) mod C, built bit by bit
#pragma unroll
        for (int q = 0; q < C; ++q) nxt[q] = obs_sel((r & bit) != 0, cur[(q + bit) % C], cur[q]);
#pragma unroll
        for (int q = 0; q < C; ++q) cur[q] = nxt[q];
    }
#pragma unroll
    for (int q = 0; q < C; ++q) {
        int j = q + r;
        if (j >= C) j -= C;
        *reinterpret_cast<ulonglong2*>(dst + 16 * j) = make_ulonglong2(cur[q].lo, cur[q].hi);
    }
}
#endif

// Shared-memory views of ONE tile for ONE period (all regions laid out like the global arrays: [E][m] etc.).
struct TileSmem {
    const void* act;            // [E][m] actions of this period, float64 or float32, then (float32 only) a [E][m] float64 scratch
                                // for the shared reward (see tile_period; float64 actions are overwritten by it once consumed)
    const int32_t* dem;         // [R][E] customer demand of this period
    int32_t *inv, *bl, *ou, *pipe, *hd, *ho, *carry, *bt;   // state, updated in place
    unsigned char* obs;         // [E][m][O] observation tile (float64, float32 or bfloat16)
    double* rew;                // [E][m] / [E] reward tile
    double* prof;               // [E][m] profits of the period, or null (episode kernel with evaluation accumulators)
    double* ret;                // [E][m] / [E] episode returns, or null (episode kernel): reward added in place, period by period
};

// Per-thread constants of the lanes = stages mapping.
template <int MAXC>
struct LaneCtx {
    NodeParams np;
    int child_lane[MAXC];
    const double* tabrow;
    int lane, i, tbase, e_loc, cell;
    bool ok, is_last;
};

template <int M_PAD, int MAXC, bool DIV>
__device__ __forceinline__ LaneCtx<MAXC> make_lane_ctx(const StepArgs& A, int tid) {
    constexpr int EPW = 32 / M_PAD;
    LaneCtx<MAXC> L;
    L.lane = tid & 31;
    L.i = L.lane % M_PAD;                             // stage / node of this lane
    const int sub = L.lane / M_PAD;                   // env slot inside the warp
    L.tbase = L.lane - L.i;                           // first lane of this env's tile
    L.e_loc = (tid >> 5) * EPW + sub;                 // env inside the CTA tile
    const int m = KF(m);
    L.ok = L.i < m && sub < EPW;                      // full tiles only: every env slot is live
    L.cell = L.e_loc * m + L.i;                       // index inside a [E][m] tile
    L.np = load_node(A.nodes + (L.ok ? L.i : 0));
    if constexpr (DIV) {
#pragma unroll
        for (int k = 0; k < MAXC; ++k) L.child_lane[k] = L.ok ? child_lane_of(L.np, k) : -1;
    } else {
#pragma unroll
        for (int k = 0; k < MAXC; ++k) L.child_lane[k] = -1;
    }
    L.is_last = (L.i == m - 1);
    L.tabrow = KHAS(tab) ? A.tab + (size_t)(L.ok ? L.i : 0) * 4 * KF(TL) : nullptr;
    return L;
}


// ONE period of ONE tile out of shared memory: read the lane's cell, the period's arithmetic (identical to step_kernel),
// write the new state in place and the observation / reward tiles.  `before_store` runs between the arithmetic and the
// writes (a multi-period launch waits there for the previous period's bulk stores).  No barriers or fences in here:
// the caller orders the tile's loads before and its stores after.
//   j = period index inside the launch (diagnostics block, MANY only), t = period being simulated, n0 = first env of the tile
//   EP: episode kernel — S.dem is the tile's whole [E][R][T] trace, and the profits go to S.prof when it is set
template <int M_PAD, int DMAX, int PMAX, int MAXC, bool DIV, bool MANY, bool EP = false, typename BeforeStore>
__device__ __forceinline__ void tile_period(const StepArgs& A, const TileLayout& TLY, const TileSmem& S, const LaneCtx<MAXC>& L,
                                            int t, int j, int64_t n0, bool delayed, BeforeStore&& before_store) {
    const NodeParams& np = L.np;
    const int lane = L.lane, i = L.i, tbase = L.tbase, e_loc = L.e_loc, cell = L.cell;
    const bool ok = L.ok, is_last = L.is_last;
    const int m = KF(m), O = KF(O), E = KT(E);
    const int es = obs_elem_bytes(KF(obs_type));     // observation element size
    const int delay_m1 = np.delay - 1;
    const double om_d = (double)np.order_max;
    const double* __restrict__ tabrow = L.tabrow;
    int32_t* my_pipe = S.pipe + e_loc * KF(L) + np.pipe_off;
    (void)lane; (void)E; (void)O; (void)es;
    // ---- read the tile ----------------------------------------------------------------------
    double act = 0.0;
    int inv = 0, backlog = 0, order_u = 0, carry = 0, cust = 0;
    int pipe[DMAX], hd[PMAX], ho[PMAX], bt[MAXC];
#pragma unroll
    for (int k = 0; k < DMAX; ++k) pipe[k] = 0;
#pragma unroll
    for (int jj = 0; jj < PMAX; ++jj) { hd[jj] = 0; ho[jj] = 0; }
#pragma unroll
    for (int k = 0; k < MAXC; ++k) bt[k] = 0;
    if (ok) {
        act = load_action(S.act, cell, KF(act_f32) != 0);
        inv = S.inv[cell];
        backlog = S.bl[cell];
        order_u = S.ou[cell];
#pragma unroll
        for (int k = 0; k < DMAX; ++k)
            if (k < np.delay) pipe[k] = my_pipe[k];
        if (KF(need_hd)) {
#pragma unroll
            for (int jj = 0; jj < PMAX; ++jj)
                if (jj < KF(P)) hd[jj] = S.hd[cell * KF(P) + jj];
        }
        if (KF(need_ho)) {
#pragma unroll
            for (int jj = 0; jj < PMAX; ++jj)
                if (jj < KF(P)) ho[jj] = S.ho[cell * KF(P) + jj];
        }
        if (np.retailer_idx >= 0) cust = EP ? S.dem[(e_loc * KF(R) + np.retailer_idx) * KF(T) + t] : S.dem[np.retailer_idx * E + e_loc];
        if (KF(has_carry)) carry = S.carry[cell];
        if constexpr (DIV) {
            if (np.bt_off >= 0) {
#pragma unroll
                for (int k = 0; k < MAXC; ++k)
                    if (k < np.nchild) bt[k] = S.bt[e_loc * KF(NB) + np.bt_off + k];
            }
        }
    }

    // ---- one period (identical arithmetic to step_kernel) --------------------------------------
    const int order = ok ? decode_order(act, om_d, KF(std_actions) != 0, KF(multi) != 0, A.a, A.bma, A.inv_bma, KBMA_POW2) : 0;
    int demand;
    int od[MAXC];
    if constexpr (DIV) {
        int sum = 0;
#pragma unroll
        for (int k = 0; k < MAXC; ++k) {
            od[k] = 0;
            if (k < KF(maxc)) {
                const int v = __shfl_sync(0xffffffffu, order, tbase + (L.child_lane[k] < 0 ? 0 : L.child_lane[k]));
                od[k] = L.child_lane[k] < 0 ? 0 : v;
                sum += od[k];
            }
        }
        demand = (np.retailer_idx >= 0) ? min(cust, np.inv_max) : sum;
    } else {
        const int down = __shfl_up_sync(0xffffffffu, order, 1);
        demand = (i == 0) ? min(cust, np.inv_max) : down;
    }
    int acq = carry;
    int carry_new = 0;
    if (t >= np.delay) {
        acq += pipe[0];
        if (delayed && t < KF(T) - 1) { carry_new = acq; acq = 0; }
    }
    const int ship = min(backlog + demand, inv + acq);
    int incoming;
    int err_code = 0;
    if constexpr (DIV) {
        int st[MAXC];
#pragma unroll
        for (int k = 0; k < MAXC; ++k) st[k] = 0;
        if (ok && np.nchild == 1) st[0] = ship;
        if (ok && np.nchild > 1)
            err_code = split_ship<MAXC>(np.nchild, ship, demand, backlog, np.demand_max, KF(wd_mult1), KF(wd_mult), od, bt, st);
        incoming = order;
#pragma unroll
        for (int k = 0; k < MAXC; ++k) {
            if (k < KF(maxc)) {
                const int v = __shfl_sync(0xffffffffu, st[k], tbase + (np.parent < 0 ? 0 : np.parent));
                if (np.parent >= 0 && np.child_slot == k) incoming = v;
            }
        }
    } else {
        const int up = __shfl_down_sync(0xffffffffu, ship, 1);
        incoming = is_last ? order : up;
    }
    int backlog_new = backlog + demand - ship;
    if (KF(cap_backlog)) backlog_new = min(backlog_new, np.demand_max);
    const int order_u_new = min(max(order_u + order - acq, 0), np.inv_max);
    const int inv_new = min(max(inv + acq - ship, 0), np.inv_max);
#pragma unroll
    for (int k = 0; k < DMAX; ++k) {
        const int nxt = (k + 1 < DMAX) ? pipe[k + 1] : 0;
        pipe[k] = (k == delay_m1) ? incoming : nxt;
    }
#pragma unroll
    for (int jj = PMAX - 1; jj > 0; --jj) { hd[jj] = hd[jj - 1]; ho[jj] = ho[jj - 1]; }
    hd[0] = demand;
    ho[0] = order;

    const double profit = ok ? profit_of(np.p, np.c, np.h, np.bc, np.target, ship, order, inv_new, backlog_new) : 0.0;
    double reward_out;
    if (KF(multi)) {
        if (KF(independent)) {
            reward_out = profit;
        } else if (!(MANY && (m >= 6 || !KHAS(obs)))) {
            // shared reward by shuffles: measured faster for the plain step kernels and for 4-wide chains
            reward_out = div_by_m(tile_seq_sum<M_PAD>(profit, m, tbase), m, A.inv_m, KM_POW2);
        } else {
            // multi-period kernels of wider networks (8-stage 0.90 -> 0.96 of peak) and the rewards-only replay (+7-12 %):
            // shared reward: the env's m profits meet in ITS row of a [E][m] float64 scratch in this period's ACTION region,
            // refilled only after the CTA barrier below — one 8-byte store per lane, then 16-byte broadcast loads, instead of
            // 2 m shuffles.  float64 actions: the scratch IS the action tile (slot `cell` holds only this lane's action, already
            // read).  float32 actions: slot `cell` would cover the actions of cells 2 cell and 2 cell + 1, which other warps may
            // not have read yet, so the scratch sits behind the E*m*4 bytes of actions (the region is E*m*12 bytes then)
            double* scratch = reinterpret_cast<double*>(const_cast<unsigned char*>(static_cast<const unsigned char*>(S.act)) +
                                                        (KF(act_f32) ? (size_t)E * m * 4 : (size_t)0));
            if (ok) scratch[cell] = profit;
            __syncwarp();
            const double* row = scratch + e_loc * m;
            double sum = 0.0;                        // reward_sum starts at 0 and adds in stage order (MAIM_env.py:418-426)
            if ((m & 1) == 0) {
                for (int q = 0; q < m / 2; ++q) {
                    const double2 pq = reinterpret_cast<const double2*>(row)[q];
                    sum = __dadd_rn(__dadd_rn(sum, pq.x), pq.y);
                }
            } else {
                for (int q = 0; q < m; ++q) sum = __dadd_rn(sum, row[q]);
            }
            reward_out = div_by_m(sum, m, A.inv_m, KM_POW2);
        }
    } else {
        reward_out = tile_np_sum<M_PAD>(profit, m, tbase);
    }

    // ---- write the tile back (in place) ----------------------------------------------------------
    before_store();                                  // e.g. the previous period's bulk stores must be done reading the output buffer
    if (ok) {
        S.inv[cell] = inv_new;
        S.bl[cell] = backlog_new;
        S.ou[cell] = order_u_new;
#pragma unroll
        for (int k = 0; k < DMAX; ++k)
            if (k < np.delay) my_pipe[k] = pipe[k];
        if (KF(need_hd)) {
#pragma unroll
            for (int jj = 0; jj < PMAX; ++jj)
                if (jj < KF(P)) S.hd[cell * KF(P) + jj] = hd[jj];
        }
        if (KF(need_ho)) {
#pragma unroll
            for (int jj = 0; jj < PMAX; ++jj)
                if (jj < KF(P)) S.ho[cell * KF(P) + jj] = ho[jj];
        }
        if (KF(has_carry)) S.carry[cell] = carry_new;
        if constexpr (DIV) {
            if (np.bt_off >= 0) {
#pragma unroll
                for (int k = 0; k < MAXC; ++k)
                    if (k < np.nchild) S.bt[e_loc * KF(NB) + np.bt_off + k] = bt[k];
            }
            if (err_code != 0) A.err[n0 + e_loc] = err_code;
        }
        if (KF(multi)) S.rew[cell] = reward_out;
        else if (i == 0) S.rew[e_loc] = reward_out;
        if (EP && S.prof) S.prof[cell] = profit;
        if (EP && S.ret) {                           // stats_slice_kernel<true>'s order: from 0, period by period
            if (KF(multi)) S.ret[cell] = __dadd_rn(S.ret[cell], reward_out);
            else if (i == 0) S.ret[e_loc] = __dadd_rn(S.ret[e_loc], reward_out);
        }
#ifdef IMX_OBS_ROTATE
        {
            if (KHAS(obs)) {
                // build the row in registers (typed like the output elements), then store its chunks in rotated order
                unsigned long long w[OBS_ROW_BYTES / 8];
                if (KF(obs_type) == OBS_BF16) {
                    uint16_t rowh[IMX_K_O];
                    write_obs_row<DMAX, PMAX>(rowh, A, np, i, tabrow, inv_new, backlog_new, order_u_new, pipe, hd, ho, DIV);
#pragma unroll
                    for (int k = 0; k < OBS_ROW_BYTES / 8; ++k)
                        w[k] = (unsigned long long)rowh[4 * k] | ((unsigned long long)rowh[4 * k + 1] << 16) |
                               ((unsigned long long)rowh[4 * k + 2] << 32) | ((unsigned long long)rowh[4 * k + 3] << 48);
                } else if (KF(obs_type) == OBS_F32) {
                    float rowf[IMX_K_O];
                    write_obs_row<DMAX, PMAX>(rowf, A, np, i, tabrow, inv_new, backlog_new, order_u_new, pipe, hd, ho, DIV);
#pragma unroll
                    for (int k = 0; k < OBS_ROW_BYTES / 8; ++k)
                        w[k] = (unsigned long long)__float_as_uint(rowf[2 * k]) | ((unsigned long long)__float_as_uint(rowf[2 * k + 1]) << 32);
                } else {
                    double rowd[IMX_K_O];
                    write_obs_row<DMAX, PMAX>(rowd, A, np, i, tabrow, inv_new, backlog_new, order_u_new, pipe, hd, ho, DIV);
#pragma unroll
                    for (int k = 0; k < OBS_ROW_BYTES / 8; ++k) w[k] = (unsigned long long)__double_as_longlong(rowd[k]);
                }
                store_row_rotated(S.obs + (size_t)cell * OBS_ROW_BYTES, w, lane);
            }
        }
#else
        if (KHAS(obs)) write_obs_row<DMAX, PMAX>(S.obs + (size_t)cell * O * es, A, np, i, tabrow, inv_new, backlog_new, order_u_new, pipe, hd, ho, DIV);
#endif
        // optional diagnostics go straight to global memory (off the fast path)
        if (KF(has_info)) {
        const int64_t gcell = (int64_t)j * A.N * m + (n0 + e_loc) * m + i;      // [periods][N][m] blocks in a multi-period launch
        if (A.info.demand_dev) A.info.demand_dev[gcell] = demand;
        if (A.info.ship_dev) A.info.ship_dev[gcell] = ship;
        if (A.info.acquisition_dev) A.info.acquisition_dev[gcell] = acq;
        if (A.info.order_dev) A.info.order_dev[gcell] = order;
        if (A.info.profit_dev) A.info.profit_dev[gcell] = profit;
        }
    }
}

// Centralised-critic rows of one tile (imx_step_cc): lane (env e, agent i) assembles
//     [ opponent actions (m-1) | opponent observations (m-1)*O | own observation O ]        models/CC_Model.py:196-214
// from the observation tile the step has just written (all m rows of an env are written by lanes of ONE warp: the caller
// separates the two phases with __syncwarp) and from the action tile of this period (FillInActions :165-193 /
// CC_inv_management.py:516-528: opponent actions clipped to [lo, hi]; zeros at sampling time).  Opponents in agent order.
template <int BYTES> struct CcWord { typedef uint32_t type; };
template <> struct CcWord<8> { typedef unsigned long long type; };
template <> struct CcWord<2> { typedef uint16_t type; };
template <typename ObsT, int MAXC>
__device__ __forceinline__ void cc_build_row(const StepArgs& A, const TileSmem& S, unsigned char* cc_tile, const LaneCtx<MAXC>& L) {
    if (!L.ok) return;
    const int m = KF(m), O = KF(O);
    const int W = (m - 1) * (1 + O) + O;
    const int e0 = L.e_loc * m;
    // a row is copied in units of its element type (4-byte words for float32 rows, which are only 4-byte aligned — W is odd
    // for m = 2; 8-byte words for float64 rows: 17 STS.64 instead of 34 STS.32 per lane, conflict-free at a stride of 2 W words;
    // 2-byte elements for bfloat16 rows, ObsT = uint16_t, the bit patterns)
    using WordT = typename CcWord<sizeof(ObsT)>::type;
    WordT* row = reinterpret_cast<WordT*>(cc_tile) + (size_t)L.cell * W;
    const WordT* ob = reinterpret_cast<const WordT*>(S.obs);
    constexpr int VEC = 16 / sizeof(ObsT);           // elements per 16-byte shared-memory load
    // opponents in agent order without a divergent branch: the q-th opponent of agent i is j = q + (q >= i), so every lane of
    // the warp runs the same instruction stream and (specialised build: m is a literal) the loops unroll into static offsets
    int k = 0;
#pragma unroll
    for (int q = 0; q < m - 1; ++q) {
        const int j = q + (q >= L.i ? 1 : 0);
        const double v = A.cc_fill ? fmin(fmax(load_action(S.act, e0 + j, KF(act_f32) != 0), A.cc_lo), A.cc_hi) : 0.0;
        if constexpr (sizeof(ObsT) == 2) row[k++] = f32_to_bf16((float)v);
        else if constexpr (sizeof(ObsT) == 4) row[k++] = __float_as_uint((float)v);
        else row[k++] = (unsigned long long)__double_as_longlong(v);
    }
    // observation rows: 16-byte shared-memory loads where the rows are 16-byte multiples (one wavefront per quarter-warp instead
    // of the 8-way conflicts of scalar loads at a row stride of 32 or 64 bytes), element-wise stores into the critic row
    auto copy_row = [&](int cell_src) {
        const WordT* src = ob + (size_t)cell_src * O;
        if (sizeof(ObsT) > 2 && O % VEC == 0) {
#pragma unroll
            for (int q = 0; q < O / VEC; ++q) {
                if constexpr (sizeof(ObsT) == 4) {
                    const uint4 v = reinterpret_cast<const uint4*>(src)[q];
                    row[k] = v.x; row[k + 1] = v.y; row[k + 2] = v.z; row[k + 3] = v.w;
                } else if constexpr (sizeof(ObsT) == 8) {
                    const ulonglong2 v = reinterpret_cast<const ulonglong2*>(src)[q];
                    row[k] = v.x; row[k + 1] = v.y;
                }
                k += VEC;
            }
        } else {
#pragma unroll
            for (int q = 0; q < O; ++q) row[k++] = src[q];
        }
    };
#pragma unroll
    for (int q = 0; q < m - 1; ++q) copy_row(e0 + q + (q >= L.i ? 1 : 0));
    copy_row(L.cell);
}
template <int MAXC>
__device__ __forceinline__ void cc_build(const StepArgs& A, const TileLayout& TLY, const TileSmem& S, unsigned char* tile_base, const LaneCtx<MAXC>& L,
                                         int nthreads) {
    (void)nthreads;
    __syncwarp();                                    // the env's m observation rows are complete
    if (KF(obs_type) == OBS_BF16) cc_build_row<uint16_t, MAXC>(A, S, tile_base + KT(off_cc), L);
    else if (KF(obs_type) == OBS_F32) cc_build_row<float, MAXC>(A, S, tile_base + KT(off_cc), L);
    else cc_build_row<double, MAXC>(A, S, tile_base + KT(off_cc), L);
}


// Env-per-thread period (runtime-specialised build, -DIMX_STEP_ET=1, networks up to 8 nodes): thread e of the CTA's compute
// group owns env e of the tile and walks over its m nodes in an unrolled loop — the network is a set of compile-time lists
// (IMX_L_*), nothing is exchanged between threads, all 32 lanes of every warp are live and the divergent split costs each warp
// its instruction stream once per 32 envs instead of once per 4.  Same arithmetic, same order, same tile layout as tile_period.
// Used for the divergent networks, whose lanes = nodes kernels are issue-bound (profiles/r2_ncu_div2_step_kernel_lanes.txt).
#if defined(IMX_JIT) && defined(IMX_STEP_ET) && IMX_STEP_ET
#define IMX_USE_STEP_ET 1
// EP: episode kernel (as in tile_period; the noisy-delay outcomes come from episode_delayed)
template <int M, int DMAX, int PMAX, int MAXC, bool DIV, bool EP = false, typename BeforeStore>
__device__ __forceinline__ void tile_period_et(const StepArgs& A, const TileLayout& TLY, const TileSmem& S, int e, int t, int64_t n0,
                                               BeforeStore&& before_store, const EpisodeArgs* EA = nullptr) {
    constexpr int INV_MAX[M] = {IMX_L_inv_max}, ORDER_MAX[M] = {IMX_L_order_max}, DEMAND_MAX[M] = {IMX_L_demand_max};
    constexpr int DELAY[M] = {IMX_L_delay}, PIPE_OFF[M] = {IMX_L_pipe_off};
    constexpr int NCHILD[M] = {IMX_L_nchild}, RETAILER[M] = {IMX_L_retailer_idx}, BT_OFF[M] = {IMX_L_bt_off};
    constexpr int CHILDREN[M * MAXC] = {IMX_L_children};
    // float64 cost constants of the nodes as bit patterns (literals: no loads, no registers)
    constexpr unsigned long long P_BITS[M] = {IMX_L_p_bits}, C_BITS[M] = {IMX_L_c_bits}, H_BITS[M] = {IMX_L_h_bits}, BC_BITS[M] = {IMX_L_bc_bits},
                                 TG_BITS[M] = {IMX_L_target_bits};
    const int E = KT(E), O = KF(O);
    const int es = obs_elem_bytes(KF(obs_type));
    const int c0 = e * M;                            // first cell of this thread's env
    int inv[M], bl[M], ou[M], cr[M], pipe[M][DMAX], hd[M][PMAX], ho[M][PMAX], bt[M][MAXC];
    int order[M], demand[M], acq[M], ship[M], incoming[M];
    // ---- read the env out of the tile -----------------------------------------------------------------------------------
#pragma unroll
    for (int j = 0; j < M; ++j) {
        inv[j] = S.inv[c0 + j]; bl[j] = S.bl[c0 + j]; ou[j] = S.ou[c0 + j];
        cr[j] = KF(has_carry) ? S.carry[c0 + j] : 0;
#pragma unroll
        for (int k = 0; k < DMAX; ++k) pipe[j][k] = (k < DELAY[j]) ? S.pipe[e * KF(L) + PIPE_OFF[j] + k] : 0;
#pragma unroll
        for (int q = 0; q < PMAX; ++q) {
            hd[j][q] = (KF(need_hd) && q < KF(P)) ? S.hd[(c0 + j) * KF(P) + q] : 0;
            ho[j][q] = (KF(need_ho) && q < KF(P)) ? S.ho[(c0 + j) * KF(P) + q] : 0;
        }
#pragma unroll
        for (int k = 0; k < MAXC; ++k) bt[j][k] = (DIV && NCHILD[j] > 1 && k < NCHILD[j]) ? S.bt[e * KF(NB) + BT_OFF[j] + k] : 0;
        order[j] = decode_order(load_action(S.act, c0 + j, KF(act_f32) != 0), (double)ORDER_MAX[j], KF(std_actions) != 0, KF(multi) != 0, A.a, A.bma, A.inv_bma, KBMA_POW2);
    }
    // ---- demand propagation, acquisition, shipment ------------------------------------------------------------------------
#pragma unroll
    for (int j = 0; j < M; ++j) {
        if (RETAILER[j] >= 0) {
            demand[j] = min(EP ? S.dem[(e * KF(R) + RETAILER[j]) * KF(T) + t] : S.dem[RETAILER[j] * E + e], INV_MAX[j]);
        } else if (DIV) {
            int sum = 0;
#pragma unroll
            for (int k = 0; k < MAXC; ++k)
                if (k < NCHILD[j]) sum += order[CHILDREN[j * MAXC + k] >= 0 ? CHILDREN[j * MAXC + k] : 0];
            demand[j] = sum;
        } else {
            demand[j] = order[j > 0 ? j - 1 : 0];
        }
        int a = cr[j];
        cr[j] = 0;
        if (t >= DELAY[j]) {
            a += pipe[j][0];
            if (KF(noisy)) {                         // noisy delay (MAIM_env.py:449-457): hold this period's arrival back by one period
                if (t < KF(T) - 1 && (EP ? episode_delayed(*EA, n0 + e, M, KF(T), j, t) : A.mask_T[((int64_t)t * A.N + n0 + e) * M + j] != 0)) {
                    cr[j] = a;
                    a = 0;
                }
            }
        }
        acq[j] = a;
        ship[j] = min(bl[j] + demand[j], inv[j] + a);
    }
    int err_code = 0;
    if constexpr (DIV) {
        incoming[0] = order[0];
#pragma unroll
        for (int j = 0; j < M; ++j) {
            if (NCHILD[j] == 1) {
                incoming[CHILDREN[j * MAXC] >= 0 ? CHILDREN[j * MAXC] : 0] = ship[j];
            } else if (NCHILD[j] > 1) {
                int od[MAXC], st[MAXC];
#pragma unroll
                for (int k = 0; k < MAXC; ++k) od[k] = (k < NCHILD[j]) ? order[CHILDREN[j * MAXC + k] >= 0 ? CHILDREN[j * MAXC + k] : 0] : 0;
                const int code = split_ship<MAXC>(NCHILD[j], ship[j], demand[j], bl[j], DEMAND_MAX[j], KF(wd_mult1), KF(wd_mult), od, bt[j], st);
                if (code != 0 && err_code == 0) err_code = code;
#pragma unroll
                for (int k = 0; k < MAXC; ++k)
                    if (k < NCHILD[j]) incoming[CHILDREN[j * MAXC + k] >= 0 ? CHILDREN[j * MAXC + k] : 0] = st[k];
            }
        }
    } else {
#pragma unroll
        for (int j = 0; j < M; ++j) incoming[j] = (j == M - 1) ? order[j] : ship[j + 1 < M ? j + 1 : j];
    }
    // ---- state update, profit, reward ---------------------------------------------------------------------------------------
    double profit[M];
#pragma unroll
    for (int j = 0; j < M; ++j) {
        int b = bl[j] + demand[j] - ship[j];
        if (KF(cap_backlog)) b = min(b, DEMAND_MAX[j]);
        ou[j] = min(max(ou[j] + order[j] - acq[j], 0), INV_MAX[j]);
        inv[j] = min(max(inv[j] + acq[j] - ship[j], 0), INV_MAX[j]);
        bl[j] = b;
#pragma unroll
        for (int k = 0; k < DMAX; ++k) {
            const int nxt = (k + 1 < DMAX) ? pipe[j][k + 1] : 0;
            pipe[j][k] = (k == DELAY[j] - 1) ? incoming[j] : nxt;
        }
#pragma unroll
        for (int q = PMAX - 1; q > 0; --q) { hd[j][q] = hd[j][q - 1]; ho[j][q] = ho[j][q - 1]; }
        hd[j][0] = demand[j];
        ho[j][0] = order[j];
        profit[j] = profit_of(__longlong_as_double((long long)P_BITS[j]), __longlong_as_double((long long)C_BITS[j]),
                              __longlong_as_double((long long)H_BITS[j]), __longlong_as_double((long long)BC_BITS[j]),
                              __longlong_as_double((long long)TG_BITS[j]), ship[j], order[j], inv[j], bl[j]);
    }
    double reward[M];
    if (KF(multi)) {
        if (KF(independent)) {
#pragma unroll
            for (int j = 0; j < M; ++j) reward[j] = profit[j];
        } else {
            double sum = 0.0;
#pragma unroll
            for (int j = 0; j < M; ++j) sum = __dadd_rn(sum, profit[j]);
            const double r = div_by_m(sum, M, A.inv_m, KM_POW2);
#pragma unroll
            for (int j = 0; j < M; ++j) reward[j] = r;
        }
    } else {
        double r;
        if constexpr (M < 8) {
            r = 0.0;
#pragma unroll
            for (int j = 0; j < M; ++j) r = __dadd_rn(r, profit[j]);
        } else {
            r = __dadd_rn(__dadd_rn(__dadd_rn(profit[0], profit[1]), __dadd_rn(profit[2], profit[3])),
                          __dadd_rn(__dadd_rn(profit[4], profit[5]), __dadd_rn(profit[6], profit[7])));
        }
        reward[0] = r;
    }
    // ---- write the tile back ----------------------------------------------------------------------------------------------
    before_store();
#pragma unroll
    for (int j = 0; j < M; ++j) {
        S.inv[c0 + j] = inv[j]; S.bl[c0 + j] = bl[j]; S.ou[c0 + j] = ou[j];
        if (KF(has_carry)) S.carry[c0 + j] = cr[j];
#pragma unroll
        for (int k = 0; k < DMAX; ++k)
            if (k < DELAY[j]) S.pipe[e * KF(L) + PIPE_OFF[j] + k] = pipe[j][k];
#pragma unroll
        for (int q = 0; q < PMAX; ++q) {
            if (KF(need_hd) && q < KF(P)) S.hd[(c0 + j) * KF(P) + q] = hd[j][q];
            if (KF(need_ho) && q < KF(P)) S.ho[(c0 + j) * KF(P) + q] = ho[j][q];
        }
        if (DIV && NCHILD[j] > 1) {
#pragma unroll
            for (int k = 0; k < MAXC; ++k)
                if (k < NCHILD[j]) S.bt[e * KF(NB) + BT_OFF[j] + k] = bt[j][k];
        }
        if (KF(multi)) S.rew[c0 + j] = reward[j];
        if (EP && S.prof) S.prof[c0 + j] = profit[j];
        if (KHAS(obs)) {
            NodeParams np;                           // the integer maxima write_obs_row scales with (compile-time values)
            np.inv_max = INV_MAX[j]; np.order_max = ORDER_MAX[j]; np.demand_max = DEMAND_MAX[j];
            const double* __restrict__ tabrow = KHAS(tab) ? A.tab + (size_t)j * 4 * KF(TL) : nullptr;
            write_obs_row<DMAX, PMAX>(S.obs + (size_t)(c0 + j) * O * es, A, np, j, tabrow, inv[j], bl[j], ou[j], pipe[j], hd[j], ho[j], DIV);
        }
    }
    if (!KF(multi)) S.rew[e] = reward[0];
    if (EP && S.ret) {                               // stats_slice_kernel<true>'s order: from 0, period by period
#pragma unroll
        for (int j = 0; j < (KF(multi) ? M : 1); ++j) S.ret[e * (KF(multi) ? M : 1) + j] = __dadd_rn(S.ret[e * (KF(multi) ? M : 1) + j], reward[j]);
    }
    if (DIV && err_code != 0) A.err[n0 + e] = err_code;
}
#else
#define IMX_USE_STEP_ET 0
#endif

// Episode kernel with evaluation accumulators, after each period: thread e repeats eval_accumulate_kernel's float64 operations
// in its order on the observation elements the step writes (obs[i][0] = inventory, obs[i][1] = backlog: rounded to the
// observation element type and widened back) and on the period's profits.
__device__ __forceinline__ void episode_env_pass(const StepArgs& A, const TileLayout& TLY, const EpisodeArgs& EA, unsigned char* smem, int e) {
    const int m = KF(m);
    const int cols = KF(multi) ? m : 1;
    const double* rew = reinterpret_cast<const double*>(smem + KT(off_rew)) + e * cols;
    {
        double* row = reinterpret_cast<double*>(smem + EA.off_eval) + e * (4 + m);
        const int32_t* inv = reinterpret_cast<const int32_t*>(smem + KT(off_inv)) + e * m;
        const int32_t* bl = reinterpret_cast<const int32_t*>(smem + KT(off_bl)) + e * m;
        const double* prof = reinterpret_cast<const double*>(smem + EA.off_prof) + e * m;
        double ep = row[0], step_inv = 0.0, step_bl = 0.0, cust = 0.0;
        if (!KF(multi)) ep = __dadd_rn(ep, rew[0]);
        for (int i = 0; i < m; ++i) {
            const double inv_max = (double)__ldg(&A.nodes[i].inv_max);
            double x0, x1;
            if (KF(std_state)) {
                const double* tabrow = KHAS(tab) ? A.tab + (size_t)i * 4 * KF(TL) : nullptr;
                x0 = scaled(KHAS(tab), tabrow, KF(TL), TAB_INV, inv[i], inv_max, A.a, A.bma);
                x1 = scaled(KHAS(tab), tabrow, KF(TL), TAB_DEM, bl[i], (double)__ldg(&A.nodes[i].demand_max), A.a, A.bma);
            } else {
                x0 = (double)inv[i];
                x1 = (double)bl[i];
            }
            x0 = obs_stored(KF(obs_type), x0);
            x1 = obs_stored(KF(obs_type), x1);
            if (EA.rescaled) {
                x0 = rev_scale_dev(x0, inv_max, A.a, A.bma);         // the loops use inv_max for BOTH fields
                x1 = rev_scale_dev(x1, inv_max, A.a, A.bma);
            }
            if (KF(multi)) ep = __dadd_rn(ep, rew[i]);
            row[4 + i] = __dadd_rn(row[4 + i], prof[i]);
            step_inv = __dadd_rn(step_inv, x0);
            step_bl = __dadd_rn(step_bl, x1);
            if (i == 0) cust = x1;
        }
        row[0] = ep;
        row[1] = __dadd_rn(row[1], step_inv);
        row[2] = __dadd_rn(row[2], step_bl);
        row[3] = __dadd_rn(row[3], cust);
    }
}

// MANY = false: one period per launch (the loop below folds away); MANY = true: A.periods periods per launch with the
// tile's state resident in shared memory (imx_step_many) — separate kernels because the loop costs registers.
// EPISODE (with MANY): a whole episode from period 0 (imx_replay_episode) — the state starts as reset_kernel writes it instead
// of being loaded, the tile's demand trace is resident for the whole episode, rewards are stored only when A.reward is set,
// and returns / evaluation accumulators are kept in shared memory and stored once.
template <int M_PAD, int DMAX, int PMAX, int MAXC, bool DIV, bool MANY, bool EPISODE = false>
__device__ __forceinline__ void step_tile(const StepArgs& A, const TileLayout& TLY, const EpisodeArgs* EA = nullptr) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t bar[2];         // bar[b]: inputs of the periods with parity b (bar[0] also the state)

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    // M_PAD is the tile width: a power of two >= m in the ahead-of-time build, exactly m in the
    // runtime-specialised build (dense packing: 32 / m envs per warp, e.g. 5 instead of 4 for m = 6)
    constexpr int EPW = 32 / M_PAD;
    const int i = lane % M_PAD;                      // stage / node of this lane
    const int sub = lane / M_PAD;                    // env slot inside the warp
    const int e_loc = (tid >> 5) * EPW + sub;        // env inside the CTA tile
    const int m = KF(m), O = KF(O), E = KT(E);
    const bool ok = i < m && sub < EPW;               // full tiles only: every env slot is live
    const int64_t n0 = (int64_t)blockIdx.x * E;      // first env of the tile
    const int K = MANY ? A.periods : 1;              // periods this launch advances

    int32_t* s_inv = reinterpret_cast<int32_t*>(smem + KT(off_inv));
    int32_t* s_bl = reinterpret_cast<int32_t*>(smem + KT(off_bl));
    int32_t* s_ou = reinterpret_cast<int32_t*>(smem + KT(off_ou));
    int32_t* s_pipe = reinterpret_cast<int32_t*>(smem + KT(off_pipe));
    int32_t* s_hd = reinterpret_cast<int32_t*>(smem + KT(off_hd));
    int32_t* s_ho = reinterpret_cast<int32_t*>(smem + KT(off_ho));
    int32_t* s_carry = reinterpret_cast<int32_t*>(smem + KT(off_carry));
    int32_t* s_bt = reinterpret_cast<int32_t*>(smem + KT(off_bt));
    const int es = obs_elem_bytes(KF(obs_type));     // observation element size
    const int aes = KF(act_f32) ? 4 : 8;             // action element size

    const uint32_t b_cell4 = (uint32_t)E * m * 4u, b_cell8 = (uint32_t)E * m * 8u, b_act = (uint32_t)E * m * aes;
    const uint32_t b_pipe = (uint32_t)E * KF(L) * 4u, b_hist = b_cell4 * (uint32_t)KF(P);
    const uint32_t b_bt = (uint32_t)E * KF(NB) * 4u, b_dem = (uint32_t)E * 4u;
    // per-period inputs: actions + demand rows (the episode kernel's demand is resident for the whole launch)
    const uint32_t b_in = b_act + (EPISODE ? 0u : (uint32_t)KF(R) * b_dem);
    const uint32_t b_edem = (uint32_t)E * KF(R) * KF(T) * 4u;     // the tile's [E][R][T] trace (episode kernel)

    // per-period inputs of period j (actions block j, demand rows of period t0 + j) into input buffer j & 1
    auto load_inputs = [&](int j) {
        unsigned char* sa = smem + ((j & 1) ? KT(off_act2) : KT(off_act));
        int32_t* sd = reinterpret_cast<int32_t*>(smem + ((j & 1) ? KT(off_dem2) : KT(off_dem)));
        bulk_load_g2s(sa, reinterpret_cast<const unsigned char*>(A.actions) + ((int64_t)j * A.act_stride + n0 * m) * aes, b_act, &bar[j & 1]);
        if (!EPISODE)
            for (int r = 0; r < KF(R); ++r)
                bulk_load_g2s(sd + r * E, A.demand_T + ((int64_t)(A.t + j) * KF(R) + r) * A.N + n0, b_dem, &bar[j & 1]);
    };

    pdl_launch_dependents();
    if (tid == 0) {                                  // on the critical path of the tile: one barrier for a plain step
        mbar_init(&bar[0], 1);
        if (MANY) mbar_init(&bar[1], 1);
        mbar_init_fence();
    }
    __syncthreads();
    if (tid == 0) {
#if defined(IMX_JIT) && !defined(IMX_NO_ACT_PREFETCH)
        bulk_prefetch_l2(reinterpret_cast<const unsigned char*>(A.actions) + n0 * m * aes, b_act);
        if (!EPISODE)
            for (int r = 0; r < KF(R); ++r) bulk_prefetch_l2(A.demand_T + ((int64_t)A.t * KF(R) + r) * A.N + n0, b_dem);
#endif
        pdl_wait();                                  // state written by the previous step must be complete and visible
        if (EPISODE) {                               // no state to load: the actions of period 0 (+ the replayed trace)
            mbar_expect_tx(&bar[0], b_in + (EA->demand ? b_edem : 0u));
            load_inputs(0);
            if (EA->demand) bulk_load_g2s(smem + EA->off_edem, EA->demand + n0 * KF(R) * KF(T), b_edem, &bar[0]);
        } else {
        uint32_t bytes = b_in + 3u * b_cell4 + b_pipe;
        if (KF(need_hd)) bytes += b_hist;
        if (KF(need_ho)) bytes += b_hist;
        if (KF(has_carry)) bytes += b_cell4;
        if (DIV && KF(NB) > 0) bytes += b_bt;
        mbar_expect_tx(&bar[0], bytes);
        load_inputs(0);
        bulk_load_g2s(s_inv, A.inv + n0 * m, b_cell4, &bar[0]);
        bulk_load_g2s(s_bl, A.backlog + n0 * m, b_cell4, &bar[0]);
        bulk_load_g2s(s_ou, A.order_u + n0 * m, b_cell4, &bar[0]);
        bulk_load_g2s(s_pipe, A.pipe + n0 * KF(L), b_pipe, &bar[0]);
        if (KF(need_hd)) bulk_load_g2s(s_hd, A.hist_d + n0 * m * KF(P), b_hist, &bar[0]);
        if (KF(need_ho)) bulk_load_g2s(s_ho, A.hist_o + n0 * m * KF(P), b_hist, &bar[0]);
        if (KF(has_carry)) bulk_load_g2s(s_carry, A.carry + n0 * m, b_cell4, &bar[0]);
        if (DIV && KF(NB) > 0) bulk_load_g2s(s_bt, A.bt + n0 * KF(NB), b_bt, &bar[0]);
        }
        if (K > 1) {                                 // period 1's inputs land while period 0 computes
            mbar_expect_tx(&bar[1], b_in);
            load_inputs(1);
        }
    }

    // per-lane constants (overlaps the bulk loads)
    const LaneCtx<MAXC> L = make_lane_ctx<M_PAD, MAXC, DIV>(A, tid);
    pdl_wait();
    if (EPISODE) {
        // reset(): inv = init_inv, every other state word 0 (reset_kernel), the watchdog flags cleared, returns and accumulators
        // at 0, and a Philox trace drawn into the demand region exactly as demand_generate_kernel draws it
        const int nthr = (int)blockDim.x;
        const int state_words = (KT(off_dem) - KT(off_inv)) / 4;     // inv .. bt are consecutive regions
        for (int k = tid; k < state_words; k += nthr) s_inv[k] = (k < E * m) ? __ldg(&A.nodes[k % m].init_inv) : 0;
        double* s_acc = reinterpret_cast<double*>(smem + EA->off_ret);  // returns, then accumulators
        for (int k = tid; k < (EA->off_prof - EA->off_ret) / 8; k += nthr) s_acc[k] = 0.0;
        for (int k = tid; k < E; k += nthr) A.err[n0 + k] = 0;
        if (!EA->demand) {
            int32_t* s_d = reinterpret_cast<int32_t*>(smem + EA->off_edem);
            const int pairs = (KF(T) + 1) / 2;
            for (int k = tid; k < E * KF(R) * pairs; k += nthr) {
                const int p = k % pairs, er = k / pairs;             // er = e * R + r
                int d0, d1;
                draw_demand_pair(EA->gen, n0 + er / KF(R), er % KF(R), 2 * p, d0, d1);
                s_d[er * KF(T) + 2 * p] = d0;
                if (2 * p + 1 < KF(T)) s_d[er * KF(T) + 2 * p + 1] = d1;
            }
        }
        __syncthreads();
    }

    for (int j = 0; j < K; ++j) {
    const int t = A.t + j;                           // period being simulated
    const int b = j & 1;
    const void* s_act = smem + (b ? KT(off_act2) : KT(off_act));
    const int32_t* s_dem = reinterpret_cast<const int32_t*>(smem + (b ? KT(off_dem2) : KT(off_dem)));
    unsigned char* s_obs = smem + KT(off_obs);       // ONE output buffer: period j - 1's bulk stores have long finished
    double* s_rew = reinterpret_cast<double*>(smem + KT(off_rew));   // reading it when period j's dynamics are done (waited below)
    bool delayed = false;
    if (KF(noisy) && ok)
        delayed = EPISODE ? episode_delayed(*EA, n0 + e_loc, m, KF(T), i, t) : A.mask_T[((int64_t)t * A.N + n0 + e_loc) * m + i] != 0;

    mbar_wait(&bar[b], (uint32_t)((j >> 1) & 1));

    const TileSmem S = {s_act, EPISODE ? reinterpret_cast<const int32_t*>(smem + EA->off_edem) : s_dem, s_inv, s_bl, s_ou, s_pipe, s_hd,
                        s_ho, s_carry, s_bt, s_obs, s_rew, (EPISODE && EA->eval) ? reinterpret_cast<double*>(smem + EA->off_prof) : nullptr,
                        (EPISODE && EA->ret) ? reinterpret_cast<double*>(smem + EA->off_ret) : nullptr};
    auto before_store = [&]() {
        if (MANY && j > 0) {                         // the previous period's stores must be done reading the output buffer
            if (tid == 0) bulk_wait_read_all();
            __syncthreads();
        }
    };
#if IMX_USE_STEP_ET
    tile_period_et<IMX_K_m, DMAX, PMAX, MAXC, DIV, EPISODE>(A, TLY, S, tid, t, n0, before_store, EA);
    (void)L; (void)delayed;
#else
    tile_period<M_PAD, DMAX, PMAX, MAXC, DIV, MANY, EPISODE>(A, TLY, S, L, t, j, n0, delayed, before_store);
#endif
    if (!MANY && KHAS(cc)) cc_build<MAXC>(A, TLY, S, smem, L, (int)blockDim.x);
    fence_proxy_async_smem();          // every writer orders its generic-proxy stores before the bulk copies
    __syncthreads();                   // ... and everybody is done reading input buffer b
    if (tid == 0) {
        if (!MANY && KHAS(cc)) bulk_store_only(reinterpret_cast<unsigned char*>(A.cc) + n0 * m * A.cc_W * es, smem + KT(off_cc), (uint32_t)E * m * A.cc_W * es);
        if (KHAS(obs)) bulk_store_only(reinterpret_cast<unsigned char*>(A.obs) + (int64_t)j * A.obs_stride_bytes + n0 * m * O * es, s_obs, (uint32_t)E * m * O * es);
        if (!EPISODE || A.reward)
            bulk_store_only(A.reward + (int64_t)j * A.rew_stride + (KF(multi) ? n0 * m : n0), s_rew, KF(multi) ? b_cell8 : (uint32_t)E * 8u);
        if (j == K - 1) {              // the tile's state leaves the SM once per launch
            bulk_store_only(A.inv + n0 * m, s_inv, b_cell4);
            bulk_store_only(A.backlog + n0 * m, s_bl, b_cell4);
            bulk_store_only(A.order_u + n0 * m, s_ou, b_cell4);
            bulk_store_only(A.pipe + n0 * KF(L), s_pipe, b_pipe);
            if (KF(need_hd)) bulk_store_only(A.hist_d + n0 * m * KF(P), s_hd, b_hist);
            if (KF(need_ho)) bulk_store_only(A.hist_o + n0 * m * KF(P), s_ho, b_hist);
            if (KF(has_carry)) bulk_store_only(A.carry + n0 * m, s_carry, b_cell4);
            if (DIV && KF(NB) > 0) bulk_store_only(A.bt + n0 * KF(NB), s_bt, b_bt);
        }
        bulk_commit();
        if (j + 2 < K) {               // input buffer b is free again: fetch the inputs of period j + 2
            mbar_expect_tx(&bar[b], b_in);
            load_inputs(j + 2);
        }
    }
    // (reads this period's reward / state / profit tiles: the next period overwrites them only behind its before_store barrier)
    if (EPISODE && EA->eval && tid < E) episode_env_pass(A, TLY, *EA, smem, tid);
    }   // periods
    if (EPISODE && (EA->ret || EA->eval)) {      // returns and accumulator rows leave the SM once per episode
        fence_proxy_async_smem();
        __syncthreads();
        if (tid == 0) {
            const int cols = KF(multi) ? m : 1;
            if (EA->ret) bulk_store_only(EA->ret + n0 * cols, smem + EA->off_ret, (uint32_t)E * cols * 8u);
            if (EA->eval) bulk_store_only(EA->eval + n0 * (4 + m), smem + EA->off_eval, (uint32_t)E * (4 + m) * 8u);
            bulk_commit();
        }
    }
    if (tid == 0) bulk_wait_read_all();  // shared memory must outlive the bulk engine's reads
}

// One period per launch (step()).
#if defined(IMX_JIT) && defined(IMX_STEP_MAXNREG)
#define IMX_STEP_BOUNDS __maxnreg__(IMX_STEP_MAXNREG)            /* experiment knob of the specialised build (host: IMX_STEP_MAXNREG) */
#else
#define IMX_STEP_BOUNDS __launch_bounds__(TMA_THREADS)
#endif
template <int M_PAD, int DMAX, int PMAX, int MAXC, bool DIV>
__global__ void IMX_STEP_BOUNDS step_kernel_tma(const __grid_constant__ StepArgs A, const __grid_constant__ TileLayout TLY) {
    step_tile<M_PAD, DMAX, PMAX, MAXC, DIV, false>(A, TLY);
}

// A.periods periods per launch (imx_step_many).  The runtime-specialised build bounds its registers (IMX_MANY_MAXNREG,
// set by the host; measured: the loop wants 40-70, a cap at 32 spills and loses 13 %).
#if defined(IMX_JIT) && defined(IMX_MANY_MAXNREG)
#define IMX_MANY_BOUNDS __maxnreg__(IMX_MANY_MAXNREG)
#elif defined(IMX_JIT)
#define IMX_MANY_BOUNDS __launch_bounds__(TMA_THREADS, 1)
#else
#define IMX_MANY_BOUNDS __launch_bounds__(TMA_THREADS)
#endif
template <int M_PAD, int DMAX, int PMAX, int MAXC, bool DIV>
__global__ void IMX_MANY_BOUNDS step_kernel_tma_many(const __grid_constant__ StepArgs A, const __grid_constant__ TileLayout TLY) {
    step_tile<M_PAD, DMAX, PMAX, MAXC, DIV, true>(A, TLY);
}

// A whole stored-plan episode per launch (imx_replay_episode): reset + A.periods = T periods + returns / accumulators.
template <int M_PAD, int DMAX, int PMAX, int MAXC, bool DIV>
__global__ void IMX_MANY_BOUNDS step_kernel_tma_episode(const __grid_constant__ StepArgs A, const __grid_constant__ TileLayout TLY,
                                                        const __grid_constant__ EpisodeArgs EA) {
    step_tile<M_PAD, DMAX, PMAX, MAXC, DIV, true, true>(A, TLY, &EA);
}

}  // namespace imx
