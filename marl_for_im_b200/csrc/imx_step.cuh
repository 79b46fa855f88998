// imx_step.cuh — the single-period environment step kernel (serial and divergent networks).
//
// Mapping: lanes = stages.  A warp is cut into tiles of M_PAD lanes (M_PAD = m rounded up to a
// power of two); one tile simulates one environment, lane i of the tile owns stage / node i.
// The only cross-stage dependencies of a period are resolved with warp shuffles inside the tile:
//   serial     demand_i = order_{i-1}   (shfl_up)     pipeline input_i = ship_{i+1}  (shfl_down)
//   divergent  demand_i = sum of the children's orders (gather)   pipeline input_i = ship_to[parent -> i] (scatter)
// Restates: MAIM_env.py:330-436 + :242-328, IM_env.py:231-374, MAIM_div_env.py:441-655 + :343-439,
// IM_div_env.py:304-563 (see SURVEY.md appendix A for the state-machine form).
//
// Memory: state is int32 structure-of-arrays [N][m] per field (the tile's lanes read consecutive
// words → every warp-level request is one contiguous 128-byte line), the ragged pipeline record
// is [N][L].  Observations ([N][m][O] float64, 60 % of all traffic) are staged per warp in shared
// memory and leave the SM as ONE TMA bulk copy per warp (cp.async.bulk shared→global).
#pragma once

#include "imx_device.cuh"

namespace imx {

constexpr int STEP_THREADS = 256;

// np.sum order for the IM kinds' scalar reward (numpy pairwise_sum: sequential below 8 elements,
// eight running accumulators from 8 to 128) — IM_env.py:372, IM_div_env.py:561.
template <int M_PAD>
__device__ __forceinline__ double tile_np_sum(double v, int m, int tb) {
    if constexpr (M_PAD < 8) {
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < M_PAD; ++j) {
            const double x = __shfl_sync(0xffffffffu, v, tb + (j));
            if (j < m) s = __dadd_rn(s, x);
        }
        return s;
    } else {
        if (m < 8) {
            double s = 0.0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const double x = __shfl_sync(0xffffffffu, v, tb + (j));
                if (j < m) s = __dadd_rn(s, x);
            }
            return s;
        }
        double r[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = __shfl_sync(0xffffffffu, v, tb + (j));
        const int full = m - (m % 8);
#pragma unroll
        for (int base = 8; base < M_PAD; base += 8) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const double x = __shfl_sync(0xffffffffu, v, tb + (base + j));
                if (base + j < full) r[j] = __dadd_rn(r[j], x);
            }
        }
        double s = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                             __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
#pragma unroll
        for (int j = 8; j < M_PAD; ++j) {
            const double x = __shfl_sync(0xffffffffu, v, tb + (j));
            if (j >= full && j < m) s = __dadd_rn(s, x);
        }
        return s;
    }
}

// MAIM shared reward: reward_sum starts at integer 0 and adds the profits in stage order
// (MAIM_env.py:418-426), then / num_stages (:434).
template <int M_PAD>
__device__ __forceinline__ double tile_seq_sum(double v, int m, int tb) {
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < M_PAD; ++j) {
        const double x = __shfl_sync(0xffffffffu, v, tb + (j));
        if (j < m) s = __dadd_rn(s, x);
    }
    return s;
}

// The same sum with the tile's profits exchanged through shared memory instead of shuffles (the rollout loop: one 8-byte
// store per lane and M_PAD / 2 16-byte broadcast loads instead of 2 * M_PAD 32-bit shuffles).  `wbuf` is this warp's
// 32-double buffer of the current period parity; the caller synchronises the warp between the store and the loads.
template <int M_PAD>
__device__ __forceinline__ double tile_seq_sum_smem(const double* wbuf, int m, int tb) {
    double s = 0.0;
    if constexpr (M_PAD % 2 == 0) {
        const double2* p = reinterpret_cast<const double2*>(wbuf + tb);       // tb * 8 bytes is a multiple of 16
#pragma unroll
        for (int j = 0; j < M_PAD / 2; ++j) {
            const double2 q = p[j];
            if (2 * j < m) s = __dadd_rn(s, q.x);
            if (2 * j + 1 < m) s = __dadd_rn(s, q.y);
        }
    } else {
#pragma unroll
        for (int j = 0; j < M_PAD; ++j)
            if (j < m) s = __dadd_rn(s, wbuf[tb + j]);
    }
    return s;
}

// One period of the divergent split for a node with > 1 child — MAIM_div_env.py:483-579 /
// IM_div_env.py:403-502.  The reference hands out goods one unit per child per round-robin pass
// (whole passes: the shipped amount may go negative inside a pass, the ledger may go negative; both
// are reproduced).  Passes are applied in BATCHES: between two events (a child's counter reaching
// zero, the goods or the outstanding total running out) every pass does the same thing, so the
// number of passes up to the next event is computed in closed form and applied at once — at most
// nchild + 1 batches instead of up to demand_max passes, with identical results.  The watchdog
// counters count passes, exactly like the reference's while_counter.
// Returns the watchdog code (0 ok; 1..4 = the reference's "Infinite Loop k").
// ceil(a / b) for a >= 0 and b = a count of children in [1, MAXC], without an integer division (20+ instructions each,
// two per batch — a fifth of the divergent kernel's issue slots): b <= 2 is a shift; otherwise multiply-high with
// ceil(2^32 / b), exact while (a + b - 1) * b < 2^32 (checked: larger amounts take the division).
template <int MAXC>
__device__ __forceinline__ int ceil_div_pos(int a, int b) {
    const uint32_t x = (uint32_t)(a + b - 1);
    if constexpr (MAXC <= 2) {
        return (int)(b == 2 ? x >> 1 : x);
    } else {
        if (x >> 28) return (int)(x / (uint32_t)b);
        const uint32_t magic = b == 2 ? 0x80000000u : b == 3 ? 0x55555556u : b == 4 ? 0x40000000u : b == 5 ? 0x33333334u
                             : b == 6 ? 0x2AAAAAABu : b == 7 ? 0x24924925u : 0x20000000u;
        return (int)(b == 1 ? x : __umulhi(x, magic));
    }
}

// while sum(cnt_k) > 0 and amt > 0: for k: if cnt_k > 0: st_k++, cnt_k--, amt--       (LOOP1 / LOOP2)
template <int MAXC>
__device__ __forceinline__ int drain_round_robin(int nchild, int (&cnt)[MAXC], int (&st)[MAXC], int& amt, int limit) {
    int passes = 0;
    // every batch ends with a counter emptied, the goods gone or the total gone, so nchild batches suffice: a bounded,
    // fully unrolled loop (MAXC = 2 for div1 / div2) instead of a data-dependent back edge
#pragma unroll
    for (int it = 0; it < MAXC; ++it) {
        int sum = 0, active = 0, lo = 0x7fffffff;
#pragma unroll
        for (int k = 0; k < MAXC; ++k) {
            if (k < nchild) {
                sum += cnt[k];
                if (cnt[k] > 0) { active += 1; lo = min(lo, cnt[k]); }
            }
        }
        if (!(sum > 0 && amt > 0)) break;
        // sum > 0 implies active >= 1; identical passes until a counter empties, the goods run out or the total does
        const int p = min(lo, min(ceil_div_pos<MAXC>(amt, active), ceil_div_pos<MAXC>(sum, active)));
#pragma unroll
        for (int k = 0; k < MAXC; ++k) {
            if (k < nchild && cnt[k] > 0) { st[k] += p; cnt[k] -= p; }
        }
        amt -= p * active;
        passes += p;
        if (passes > limit) return 1;
    }
    return 0;
}

// demand_max * mult saturated at INT_MAX: demand_max may reach INT_MAX, and a pass count never exceeds the int32 amount
// it hands out, so the saturated limit fires exactly where the reference's unbounded product would
__device__ __forceinline__ int watchdog_limit(int demand_max, int mult) {
    return demand_max > 0x7fffffff / mult ? 0x7fffffff : demand_max * mult;
}

template <int MAXC>
__device__ __forceinline__ int split_ship(int nchild, int ship, int demand, int backlog, int demand_max, int mult1,
                                          int mult, const int (&od)[MAXC], int (&bt)[MAXC], int (&st)[MAXC]) {
    int amt = ship;
    const int limit1 = watchdog_limit(demand_max, mult1), limit = watchdog_limit(demand_max, mult);
#pragma unroll
    for (int k = 0; k < MAXC; ++k) st[k] = 0;

    if (ship >= demand) {
        if (backlog > 0) {
            if (drain_round_robin<MAXC>(nchild, bt, st, amt, limit1)) return 1;
            if (amt > 0 && demand > 0) {
                int out[MAXC];
#pragma unroll
                for (int k = 0; k < MAXC; ++k) out[k] = (k < nchild) ? od[k] : 0;
                if (drain_round_robin<MAXC>(nchild, out, st, amt, limit)) return 2;
#pragma unroll
                for (int k = 0; k < MAXC; ++k)
                    if (k < nchild) bt[k] += out[k];
            }
        } else {
#pragma unroll
            for (int k = 0; k < MAXC; ++k) st[k] += (k < nchild) ? od[k] : 0;
        }
    } else {
        if (backlog > 0) {
            if (drain_round_robin<MAXC>(nchild, bt, st, amt, limit)) return 3;
        } else {
            // while amt > 0: for k: if st_k < od_k + bt_k: st_k++, amt--                          (LOOP4)
            // every batch fills a child up to od_k + bt_k or hands out the rest of the goods, so at most nchild + 1 batches run:
            // the only back edge of the split that depends on the data, kept as a loop (an unrolled bound measured 1.5 % slower
            // on div2) and guarded against an empty batch, which would never end it
            int passes = 0;
            while (amt > 0) {
                int active = 0, lo = 0x7fffffff;
#pragma unroll
                for (int k = 0; k < MAXC; ++k) {
                    if (k < nchild && st[k] < od[k] + bt[k]) { active += 1; lo = min(lo, od[k] + bt[k] - st[k]); }
                }
                if (active == 0) return 4;                  // nobody can take a unit: the reference spins into its watchdog
                const int p = min(lo, ceil_div_pos<MAXC>(amt, active));
                if (p <= 0) return 4;                       // unreachable (amt, active, lo >= 1): a wrong division ends here, not in a hang
#pragma unroll
                for (int k = 0; k < MAXC; ++k) {
                    if (k < nchild && st[k] < od[k] + bt[k]) st[k] += p;
                }
                amt -= p * active;
                passes += p;
                if (passes > limit) return 4;
            }
        }
#pragma unroll
        for (int k = 0; k < MAXC; ++k) {
            if (k < nchild) bt[k] += od[k] - st[k];
        }
    }
    return 0;
}

// Writes one agent's observation vector (O doubles) — the field order and per-field maxima of
// SURVEY.md table A.5.  `row` points into the warp's shared-memory staging tile.
template <int DMAX, int PMAX, bool CHECKED = false>
__device__ __forceinline__ void write_obs_row(void* row, const StepArgs& A, const NodeParams& np, int node_idx,
                                              const double* __restrict__ tabrow, int inv, int backlog, int order_u,
                                              const int (&pipe)[DMAX], const int (&hd)[PMAX], const int (&ho)[PMAX], bool div) {
    const double a = A.a, bma = A.bma;
    const int TL = KF(TL);
    const double inv_max = (double)np.inv_max, order_max = (double)np.order_max;
    const double dem_max = (double)np.demand_max;
    const double ou_max = KF(multi) ? order_max : inv_max;   // MAIM_env.py:300 vs IM_env.py:265
    const float* __restrict__ tabrow_f = (KF(obs_f32) && KHAS(tab)) ? A.tabf + (size_t)node_idx * 4 * TL : nullptr;
    if (KF(std_state)) {
        OBS_PUT_SCALED(row, 0, CHECKED, tabrow, tabrow_f, TL, TAB_INV, inv, inv_max, a, bma);
        OBS_PUT_SCALED(row, 1, CHECKED, tabrow, tabrow_f, TL, TAB_DEM, backlog, dem_max, a, bma);
        OBS_PUT_SCALED(row, 2, CHECKED, tabrow, tabrow_f, TL, KF(multi) ? TAB_ORD : TAB_INV, order_u, ou_max, a, bma);
    } else {
        OBS_PUT_INT(row, 0, inv);
        OBS_PUT_INT(row, 1, backlog);
        OBS_PUT_INT(row, 2, order_u);
    }
    if (KF(multi) && !KF(std_state)) {
        // MAIM_env.py:319-324 (quirk 13): raw pipeline at [3:3+D] whatever the history offsets, rest stays 0
        for (int k = 3; k < KF(O); ++k) OBS_PUT(row, k, 0.0);
        if (KF(td)) {
#pragma unroll
            for (int k = 0; k < DMAX; ++k)
                if (k < KF(D)) OBS_PUT_INT(row, 3 + k, pipe[k]);
        }
        return;
    }
    int k0 = 3;
    if (KF(pd)) {
#pragma unroll
        for (int j = 0; j < PMAX; ++j)
            if (j < KF(P)) {
                if (KF(write_hd)) OBS_PUT_SCALED(row, k0 + j, CHECKED, tabrow, tabrow_f, TL, TAB_DEM, hd[j], dem_max, a, bma);
                else OBS_PUT(row, k0 + j, 0.0);             // quirk 2
            }
        k0 += KF(P);
    }
    if (KF(pa)) {
#pragma unroll
        for (int j = 0; j < PMAX; ++j)
            if (j < KF(P)) OBS_PUT_SCALED(row, k0 + j, CHECKED, tabrow, tabrow_f, TL, TAB_ORD, ho[j], order_max, a, bma);
        k0 += KF(P);
    }
    if (KF(td)) {
#pragma unroll
        for (int k = 0; k < DMAX; ++k) {
            if (k < KF(D)) {
                if (!KF(std_state)) OBS_PUT_INT(row, k0 + k, pipe[k]);                      // IM kinds, raw
                else if (div && KF(multi)) OBS_PUT_SCALED(row, k0 + k, CHECKED, tabrow, tabrow_f, TL, TAB_PIPE2, min(pipe[k], 2 * np.inv_max), 2.0 * inv_max, a, bma);   // MAIM_div_env.py:408-411
                else OBS_PUT_SCALED(row, k0 + k, CHECKED, tabrow, tabrow_f, TL, TAB_INV, pipe[k], inv_max, a, bma);
            }
        }
        k0 += KF(D);
    }
    if (KF(share_network)) OBS_PUT(row, k0, rescale((double)node_idx, (double)KF(m), a, bma));       // MAIM_div_env.py:434-435
}

// Flushes a warp's staged observation tile (`bytes` contiguous bytes, a multiple of 4) to global memory.
__device__ __forceinline__ void flush_obs_tile(void* gdst, const void* stile, uint32_t bytes, int lane) {
    const bool bulk_ok = ((bytes & 15u) == 0u) && ((reinterpret_cast<uintptr_t>(gdst) & 15u) == 0u);
    if (bulk_ok) fence_proxy_async_smem();      // every writer orders its stores before the async-proxy read
    __syncwarp();
    if (bulk_ok) {
        if (lane == 0) bulk_store_s2g(gdst, stile, bytes);
    } else {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(stile);
        uint32_t* dst = reinterpret_cast<uint32_t*>(gdst);
        for (uint32_t k = lane; k < bytes / 4u; k += 32) dst[k] = src[k];
    }
}

template <int M_PAD, int DMAX, int PMAX, int MAXC, bool DIV>
__global__ void __launch_bounds__(STEP_THREADS) step_kernel(const __grid_constant__ StepArgs A) {
    extern __shared__ __align__(16) unsigned char smem_obs[];
    constexpr int EPW = 32 / M_PAD;                 // envs per warp
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int i = lane % M_PAD;                     // stage / node owned by this lane
    const int sub = lane / M_PAD;                   // env slot inside the warp
    const int tbase = lane - i;                     // first lane of this env's tile
    const bool stage_ok = i < KF(m);
    const int m = KF(m), O = KF(O);

    const NodeParams np = load_node(A.nodes + (stage_ok ? i : 0));
    int child_lane[MAXC];
    if constexpr (DIV) {
#pragma unroll
        for (int k = 0; k < MAXC; ++k)
            child_lane[k] = stage_ok ? child_lane_of(np, k) : -1;
    }
    const bool is_last = (i == m - 1);
    const int delay_m1 = np.delay - 1;
    const double om_d = (double)np.order_max;
    const double* __restrict__ tabrow = KHAS(tab) ? A.tab + (size_t)(stage_ok ? i : 0) * 4 * KF(TL) : nullptr;

    const int es = KF(obs_f32) ? 4 : 8;                          // observation element size
    const int tile_bytes = (EPW * m * O * es + 15) & ~15;        // keep every warp's tile 16-byte aligned
    unsigned char* wtile = smem_obs + (size_t)warp * tile_bytes;
    bool tile_in_flight = false;

    const int64_t warps_in_grid = (int64_t)gridDim.x * (STEP_THREADS / 32);
    const int64_t n_warp_tiles = (A.N + EPW - 1) / EPW;
    for (int64_t wt = A.n_begin / EPW + (int64_t)blockIdx.x * (STEP_THREADS / 32) + warp; wt < n_warp_tiles; wt += warps_in_grid) {
        const int64_t n = wt * EPW + sub;
        const bool ok = stage_ok && n < A.N;
        const int64_t cell = n * m + i;

        // ---- loads (all issued before the first use) --------------------------------------
        double act = 0.0;
        int inv = 0, backlog = 0, order_u = 0, carry = 0, cust = 0;
        int pipe[DMAX], hd[PMAX], ho[PMAX];
        int bt[MAXC];
        bool delayed = false;
#pragma unroll
        for (int k = 0; k < DMAX; ++k) pipe[k] = 0;
#pragma unroll
        for (int j = 0; j < PMAX; ++j) { hd[j] = 0; ho[j] = 0; }
#pragma unroll
        for (int k = 0; k < MAXC; ++k) bt[k] = 0;
        if (ok) {
            act = A.actions[cell];
            inv = A.inv[cell];
            backlog = A.backlog[cell];
            order_u = A.order_u[cell];
            const int32_t* pp = A.pipe + n * KF(L) + np.pipe_off;
#pragma unroll
            for (int k = 0; k < DMAX; ++k)
                if (k < np.delay) pipe[k] = pp[k];
            if (KF(need_hd)) {
#pragma unroll
                for (int j = 0; j < PMAX; ++j)
                    if (j < KF(P)) hd[j] = A.hist_d[cell * KF(P) + j];
            }
            if (KF(need_ho)) {
#pragma unroll
                for (int j = 0; j < PMAX; ++j)
                    if (j < KF(P)) ho[j] = A.hist_o[cell * KF(P) + j];
            }
            if (np.retailer_idx >= 0) cust = A.demand_T[((int64_t)A.t * KF(R) + np.retailer_idx) * A.N + n];
            if (KF(has_carry)) carry = A.carry[cell];
            if (KF(noisy)) delayed = A.mask_T[((int64_t)A.t * A.N + n) * m + i] != 0;
            if constexpr (DIV) {
                if (np.bt_off >= 0) {
#pragma unroll
                    for (int k = 0; k < MAXC; ++k)
                        if (k < np.nchild) bt[k] = A.bt[n * KF(NB) + np.bt_off + k];
                }
            }
        }

        // ---- order clipping ---------------------------------------------------------------
        const int order = ok ? decode_order(act, om_d, KF(std_actions) != 0, KF(multi) != 0, A.a, A.bma, A.inv_bma, KBMA_POW2) : 0;

        // ---- demand propagation -----------------------------------------------------------
        int demand;
        int od[MAXC];
        if constexpr (DIV) {
            int s = 0;
#pragma unroll
            for (int k = 0; k < MAXC; ++k) {
                od[k] = 0;
                if (k < KF(maxc)) {
                    const int v = __shfl_sync(0xffffffffu, order, tbase + (child_lane[k] < 0 ? 0 : child_lane[k]));
                    od[k] = child_lane[k] < 0 ? 0 : v;
                    s += od[k];
                }
            }
            demand = (np.retailer_idx >= 0) ? min(cust, np.inv_max) : s;
        } else {
            const int down = __shfl_up_sync(0xffffffffu, order, 1);      // lane i-1 of the same tile (unused for i == 0)
            demand = (i == 0) ? min(cust, np.inv_max) : down;
        }

        // ---- acquisition: head of the lead-time pipeline (+ replayed noisy delay) ----------
        int acq = carry;
        int carry_new = 0;
        if (A.t >= np.delay) {
            acq += pipe[0];
            if (delayed && A.t < KF(T) - 1) { carry_new = acq; acq = 0; }
        }

        // ---- shipment and state update ----------------------------------------------------
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
            incoming = order;                                   // root: its own production order
#pragma unroll
            for (int k = 0; k < MAXC; ++k) {
                if (k < KF(maxc)) {
                    const int v = __shfl_sync(0xffffffffu, st[k], tbase + (np.parent < 0 ? 0 : np.parent));
                    if (np.parent >= 0 && np.child_slot == k) incoming = v;
                }
            }
        } else {
            const int up = __shfl_down_sync(0xffffffffu, ship, 1);        // lane i+1 of the same tile (unused for the last stage)
            incoming = is_last ? order : up;
        }

        int backlog_new = backlog + demand - ship;
        if (KF(cap_backlog)) backlog_new = min(backlog_new, np.demand_max);
        const int order_u_new = min(max(order_u + order - acq, 0), np.inv_max);
        const int inv_new = min(max(inv + acq - ship, 0), np.inv_max);
        // shift the lead-time register by one period and insert this period's shipment at slot delay-1
        // (selects, not indexed stores: the array must stay in registers)
#pragma unroll
        for (int k = 0; k < DMAX; ++k) {
            const int nxt = (k + 1 < DMAX) ? pipe[k + 1] : 0;
            pipe[k] = (k == delay_m1) ? incoming : nxt;
        }
#pragma unroll
        for (int j = PMAX - 1; j > 0; --j) { hd[j] = hd[j - 1]; ho[j] = ho[j - 1]; }
        hd[0] = demand;
        ho[0] = order;

        // ---- reward -----------------------------------------------------------------------
        const double profit = ok ? profit_of(np.p, np.c, np.h, np.bc, np.target, ship, order, inv_new, backlog_new) : 0.0;
        double reward_out;
        if (KF(multi)) {
            if (KF(independent)) reward_out = profit;
            else reward_out = div_by_m(tile_seq_sum<M_PAD>(profit, m, tbase), m, A.inv_m, KM_POW2);
        } else {
            reward_out = tile_np_sum<M_PAD>(profit, m, tbase);
        }

        // ---- stores -----------------------------------------------------------------------
        if (tile_in_flight) {                       // the previous iteration's bulk copy must have read the tile
            if (lane == 0) bulk_wait_read_all();
            __syncwarp();
            tile_in_flight = false;
        }
        if (ok) {
            A.inv[cell] = inv_new;
            A.backlog[cell] = backlog_new;
            A.order_u[cell] = order_u_new;
            int32_t* pp = A.pipe + n * KF(L) + np.pipe_off;
#pragma unroll
            for (int k = 0; k < DMAX; ++k)
                if (k < np.delay) pp[k] = pipe[k];
            if (KF(need_hd)) {
#pragma unroll
                for (int j = 0; j < PMAX; ++j)
                    if (j < KF(P)) A.hist_d[cell * KF(P) + j] = hd[j];
            }
            if (KF(need_ho)) {
#pragma unroll
                for (int j = 0; j < PMAX; ++j)
                    if (j < KF(P)) A.hist_o[cell * KF(P) + j] = ho[j];
            }
            if (KF(has_carry)) A.carry[cell] = carry_new;
            if constexpr (DIV) {
                if (np.bt_off >= 0) {
#pragma unroll
                    for (int k = 0; k < MAXC; ++k)
                        if (k < np.nchild) A.bt[n * KF(NB) + np.bt_off + k] = bt[k];
                }
                if (err_code != 0) A.err[n] = err_code;
            }
            if (KF(multi)) A.reward[cell] = reward_out;
            else if (i == 0) A.reward[n] = reward_out;
            if (KF(has_info)) {
                if (A.info.demand_dev) A.info.demand_dev[cell] = demand;
                if (A.info.ship_dev) A.info.ship_dev[cell] = ship;
                if (A.info.acquisition_dev) A.info.acquisition_dev[cell] = acq;
                if (A.info.order_dev) A.info.order_dev[cell] = order;
                if (A.info.profit_dev) A.info.profit_dev[cell] = profit;
            }
            if (KHAS(obs)) write_obs_row<DMAX, PMAX>(wtile + (size_t)(sub * m + i) * O * es, A, np, i, tabrow, inv_new, backlog_new, order_u_new, pipe, hd, ho, DIV);
        }
        if (KHAS(obs)) {
            const int64_t first = wt * EPW;
            const int envs_here = (int)min((int64_t)EPW, A.N - first);
            flush_obs_tile(reinterpret_cast<unsigned char*>(A.obs) + first * m * O * es, wtile, (uint32_t)(envs_here * m * O * es), lane);
            tile_in_flight = true;
        }
    }
    // shared memory must stay valid until the bulk engine has read it
    if (tile_in_flight && lane == 0) bulk_wait_read_all();
}

}  // namespace imx
