// imx_device.cuh — device-side parameter blocks and helpers shared by the step, reset and
// rollout kernels.  sm_100a only.
#pragma once

#ifndef __CUDACC_RTC__
#include <cuda_runtime.h>
#include <stdint.h>
#else   // NVRTC has no system headers: the fixed-width types this code uses
typedef signed char int8_t;
typedef unsigned char uint8_t;
typedef int int32_t;
typedef unsigned int uint32_t;
typedef unsigned short uint16_t;
typedef long long int64_t;
typedef unsigned long long uint64_t;
typedef unsigned long uintptr_t;
#endif

#include "../../include/imx_b200.h"

// Mode flags and sizes.  Ahead-of-time kernels read them from the kernel arguments (uniform
// branches); the runtime-specialised build (imx_jit.cuh, NVRTC) defines IMX_JIT and injects every
// one of them as a literal, so the compiler folds the branches and unrolls to the exact config.
#ifdef IMX_JIT
#define KF(name) (IMX_K_##name)
#define KT(name) (IMX_KT_##name)
#define KHAS(ptr) (IMX_K_has_##ptr)
#define KBMA_POW2 (IMX_K_bma_pow2)
#define KM_POW2 (IMX_K_m_pow2)
#define KNOISY_DEMAND(g) (IMX_K_noisy_demand)
#ifndef IMX_K_has_cc
#define IMX_K_has_cc 0
#define IMX_KT_off_cc 0
#endif
#else
#define KF(name) (A.name)
#define KT(name) (TLY.name)
#define KHAS(ptr) (A.ptr != nullptr)
#define KBMA_POW2 (A.inv_bma != 0.0)
#define KM_POW2 (A.m_pow2 != 0)
#define KNOISY_DEMAND(g) ((g).noise_thr > 0.0)
#endif

namespace imx {

// ------------------------------------------------------------------------------------
// Per-node constants.  Lives in global memory (one small table per env handle); every thread
// loads the record of ITS stage once at kernel start and keeps it in registers — the
// thread -> stage mapping is fixed for the whole grid-stride loop (lane % M_PAD).
// 96 bytes = six 16-byte loads.
// ------------------------------------------------------------------------------------
struct __align__(16) NodeParams {
    int32_t inv_max;
    int32_t order_max;
    int32_t demand_max;    // serial: = inv_max (scales backlog / demand history there)
    int32_t delay;
    int32_t pipe_off;      // first slot of this node in the ragged pipe[L] record
    int32_t init_inv;
    int32_t parent;        // divergent: lane of the parent (-1 for the root / serial)
    int32_t child_slot;    // divergent: position among the parent's children
    int32_t nchild;        // divergent: number of children
    int32_t bt_off;        // divergent: offset of this node's ledger in bt[NB] (-1: not a split node)
    int32_t retailer_idx;  // row of the demand trace feeding this node (-1: not a retailer)
    int32_t parent_nchild; // divergent: number of children of the parent (> 1: this node's inflow comes out of a split)
    double p;              // unit sell price
    double c;              // unit buy cost
    double h;              // stock holding cost
    double bc;             // backlog cost
    double target;         // inventory target
    uint32_t child_lo, child_hi;   // divergent: lanes of up to 8 children, one byte each (0xFF = none), child k in byte k
};
static_assert(sizeof(NodeParams) == 96, "NodeParams must stay 96 bytes");

// Six 16-byte read-only loads, unpacked field by field so the record stays in registers.
__device__ __forceinline__ NodeParams load_node(const NodeParams* p) {
    const int4* s = reinterpret_cast<const int4*>(p);
    const int4 q0 = __ldg(s), q1 = __ldg(s + 1), q2 = __ldg(s + 2), q3 = __ldg(s + 3), q4 = __ldg(s + 4), q5 = __ldg(s + 5);
    NodeParams n;
    n.inv_max = q0.x; n.order_max = q0.y; n.demand_max = q0.z; n.delay = q0.w;
    n.pipe_off = q1.x; n.init_inv = q1.y; n.parent = q1.z; n.child_slot = q1.w;
    n.nchild = q2.x; n.bt_off = q2.y; n.retailer_idx = q2.z; n.parent_nchild = q2.w;
    n.p = __hiloint2double(q3.y, q3.x); n.c = __hiloint2double(q3.w, q3.z);
    n.h = __hiloint2double(q4.y, q4.x); n.bc = __hiloint2double(q4.w, q4.z);
    n.target = __hiloint2double(q5.y, q5.x); n.child_lo = (uint32_t)q5.z; n.child_hi = (uint32_t)q5.w;
    return n;
}

// Lane (inside the env's tile) of child k of this node, -1 if it has fewer children.
__device__ __forceinline__ int child_lane_of(const NodeParams& n, int k) {
    const uint32_t w = (k < 4) ? n.child_lo : n.child_hi;
    const int v = (int)((w >> ((k & 3) * 8)) & 0xFFu);
    return (k < n.nchild) ? v : -1;
}

// Batch-uniform arguments (kernel parameter space → constant bank, broadcast reads).
struct StepArgs {
    // sizes
    int64_t N;
    int64_t n_begin;           // first env this launch handles (direct kernel; the TMA kernel covers [0, n_begin))
    int32_t m, T, P, D, O, L, NB, R;
    int32_t t;                 // period being simulated (0-based)
    int32_t maxc;              // max children per node (divergent)
    // mode flags (uniform branches)
    int32_t multi;             // MAIM kinds
    int32_t std_state, std_actions, cap_backlog;
    int32_t independent, share_network;
    int32_t td, pd, pa;
    int32_t write_hd;          // demand-history slots are written into obs (false in the MAIM (F,T,F) quirk)
    int32_t noisy;             // consume the delay mask this episode
    int32_t has_carry;         // carry field allocated
    int32_t need_hd, need_ho;  // history state present
    int32_t has_info;          // any imx_info_out pointer set
    int32_t obs_type;          // element type of the observations: OBS_F64, OBS_F32 (the float32 cast of the float64 value) or OBS_BF16
    int32_t act_f32;           // actions are read as float32 (widened to float64 before decoding), else float64
    int32_t wd_mult1, wd_mult;   // watchdog multipliers: LOOP1(A) and the other three
    double a, b, bma;          // bma = b - a
    double inv_bma;            // 1/(b-a) when b-a is a power of two (the division is then an exact scaling), else 0
    double inv_m;              // RN(1/m) (shared-reward mean: an exact scaling when m is a power of two, else the reciprocal of the division below)
    // tables
    int32_t TL;                // entries per rescale table row (0: no tables, compute)
    int32_t pad_tl;
    const double* __restrict__ tab;         // [m][4][TL] exact rescale results, see build_tables() in imx_api.cu
    const float* __restrict__ tabf;         // the same table rounded to float32 (obs_f32: the value is stored as loaded, no conversion in the kernel)
    const uint16_t* __restrict__ tabh;      // the float32 table rounded to bfloat16 (round to nearest even), bit patterns
    const NodeParams* __restrict__ nodes;   // [m]
    // state (SoA, int32)
    int32_t* __restrict__ inv;
    int32_t* __restrict__ backlog;
    int32_t* __restrict__ order_u;
    int32_t* __restrict__ pipe;
    int32_t* __restrict__ hist_d;
    int32_t* __restrict__ hist_o;
    int32_t* __restrict__ carry;
    int32_t* __restrict__ bt;
    int32_t* __restrict__ err;
    const int32_t* __restrict__ demand_T;   // [T][R][N]
    const uint8_t* __restrict__ mask_T;     // [T][N][m]
    // I/O
    const void* __restrict__ actions;       // [N][m] float64, or float32 when act_f32
    double* __restrict__ obs;               // [N][m][O]
    double* __restrict__ reward;            // [N][m] or [N]
    imx_info_out info;
    // multi-period replay (imx_step_many): the TMA kernel advances `periods` periods per launch with the tile's state
    // resident in shared memory; period j reads actions + j * act_stride and writes obs / reward slices j
    int32_t periods;                        // >= 1 (1 = plain step)
    int32_t m_pow2;                         // m is a power of two
    int64_t act_stride;                     // action elements between consecutive periods' action blocks
    int64_t obs_stride_bytes;               // bytes between consecutive periods' observation blocks
    int64_t rew_stride;                     // doubles between consecutive periods' reward blocks
    // centralised-critic observation emitted by the step itself (imx_step_cc; models/CC_Model.py:165-214): for every agent the
    // row [opponent actions (m-1) | opponent observations (m-1)*O | own observation O], in the observation element type
    void* __restrict__ cc;                  // [N][m][W] or nullptr
    int32_t cc_fill;                        // 1: opponent-action slots = clip(this step's actions, cc_lo, cc_hi); 0: zeros
    int32_t cc_W;                           // (m-1)*(1+O) + O
    double cc_lo, cc_hi;
};

// ------------------------------------------------------------------------------------
// Exact float64 arithmetic.  The explicit _rn intrinsics are never contracted into FMAs, so the
// result is the same sequence of IEEE-754 roundings numpy performs.
// ------------------------------------------------------------------------------------
// rescale(v, 0, vmax, a, b) = a + ((v - 0) * (b - a)) / (vmax - 0)      MAIM_env.py:497-507
__device__ __forceinline__ double rescale(double v, double vmax, double a, double bma) {
    return __dadd_rn(a, __ddiv_rn(__dmul_rn(v, bma), vmax));
}
// rev_scale(x, 0, vmax, a, b) = ((x - a) * (vmax - 0)) / (b - a) + 0    MAIM_env.py:509-519
__device__ __forceinline__ double rev_scale(double x, double vmax, double a, double bma) {
    return __ddiv_rn(__dmul_rn(__dsub_rn(x, a), vmax), bma);
}
// the evaluation loops' rev_scale with every operation of the host expression (the trailing "+ 0" turns -0 into +0):
// (((x - a) * (max - 0)) / (b - a)) + 0                                                 MAIM_env.py:509-519
__device__ __forceinline__ double rev_scale_dev(double x, double vmax, double a, double bma) {
    return __dadd_rn(__ddiv_rn(__dmul_rn(__dsub_rn(x, a), __dsub_rn(vmax, 0.0)), bma), 0.0);
}
// order clipping: MAIM kinds round then clip (MAIM_env.py:344-347), IM kinds clip then round
// (IM_env.py:300-302); rint() is round-half-to-even like np.round.
__device__ __forceinline__ int decode_order(double x, double om, bool std_actions, bool multi, double a, double bma,
                                            double inv_bma, bool bma_pow2) {
    if (std_actions) {
        // dividing by a power of two is an exact exponent shift, so the multiply gives the same bits
        if (bma_pow2) x = __dmul_rn(__dmul_rn(__dsub_rn(x, a), om), inv_bma);
        else x = rev_scale(x, om, a, bma);
    }
    // round-half-to-even then clip (MAIM) and clip then round (IM) give the same integer for an integral order_max
    // (rounding is monotone and fixes 0 and order_max), so one saturating convert + an integer clamp replaces the float64
    // rint / fmin / fmax sequence (19 instructions per lane in the rollout loop); NaN converts to 0.
    // Non-finite / huge actions: the MAIM kinds round and convert BEFORE clipping (MAIM_env.py:344-347), and on the reference's
    // x86-64 the float64 -> int64 conversion of anything >= 2^63 (and of NaN, +-inf) yields INT64_MIN, which then clips to 0 —
    // so an order >= 2^63 (high word >= 0x43E00000: also +inf and positive NaN) is 0 there, not order_max.  The IM kinds clip
    // first (IM_env.py:300-302), so +inf saturates to order_max like any large value.
    const int v = min(max(__double2int_rn(x), 0), (int)om);
    return (multi && __double2hiint(x) >= 0x43E00000) ? 0 : v;
}
// Rescaled observation value.  The integer domain of every scaled field is bounded (inventory and
// unfulfilled orders by inv_max, capped backlog and demand by demand_max, pipeline entries by
// 2*max(demand_max) + children), so the host precomputes a + (v*(b-a))/max for every v with the same
// IEEE operations and the kernel replaces an FP64 division by one cached 8-byte load.
// CHECKED (reset kernel: init_inv is an arbitrary config value and the reference does not clip it before the first
// observation): a value outside the table is computed with the three IEEE operations instead.  Unchecked (step / rollout
// kernels: every value is bounded by construction, DESIGN.md section 3.2): the index is clamped for memory safety only;
// -DIMX_DEBUG_BOUNDS turns an out-of-table value into a trap.
enum : int { TAB_INV = 0, TAB_ORD = 1, TAB_DEM = 2, TAB_PIPE2 = 3 };
template <bool CHECKED = false>
__device__ __forceinline__ double scaled(bool has_tab, const double* __restrict__ tabrow, int TL, int which, int v,
                                         double vmax, double a, double bma) {
    if (has_tab) {
        if (CHECKED) {
            if ((unsigned)v >= (unsigned)TL) return rescale((double)v, vmax, a, bma);
        }
#ifdef IMX_DEBUG_BOUNDS
        if ((unsigned)v >= (unsigned)TL) __trap();
#endif
        return __ldg(tabrow + which * TL + (int)min((unsigned)v, (unsigned)(TL - 1)));
    }
    return rescale((double)v, vmax, a, bma);
}
// mean of the shared reward: reward_sum / num_stages (MAIM_env.py:434)
__device__ __forceinline__ double div_by_m(double s, int m, double inv_m, bool m_pow2) {
    if (m_pow2) return __dmul_rn(s, inv_m);
    // Correctly rounded s / m in three instructions instead of the ~16 of the general division (which also handles
    // exponent extremes that cannot occur here): with y = RN(1/m) and q0 = RN(s * y), RN(q0 + y * RN(s - m * q0)) is the
    // correctly rounded quotient (Markstein 1990; the residual s - m * q0 is exact in an FMA).  |s| is a sum of a few
    // cost * quantity products — far from overflow, underflow and subnormals; s = 0 gives +0 like the division.
    const double q0 = __dmul_rn(s, inv_m);
    const double rem = __fma_rn(-q0, (double)m, s);
    return __fma_rn(rem, inv_m, q0);
}
// Observation element types (StepArgs.obs_type; the runtime-specialised build injects it as a literal).  bfloat16 elements are
// what torch's float64 -> bfloat16 conversion gives, which rounds through float32: round-to-nearest-even of the float32 element.
enum : int { OBS_F64 = 0, OBS_F32 = 1, OBS_BF16 = 2 };
__host__ __device__ constexpr int obs_elem_bytes(int type) { return type == OBS_BF16 ? 2 : type == OBS_F32 ? 4 : 8; }

// float32 -> bfloat16 bits, round to nearest even (one F2FP; observations are never NaN)
__device__ __forceinline__ uint16_t f32_to_bf16(float x) {
    uint16_t r;
    asm("cvt.rn.bf16.f32 %0, %1;" : "=h"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float bf16_to_f32(uint16_t u) { return __uint_as_float((uint32_t)u << 16); }
// the value an observation element of type `type` holds for the float64 value x, widened back to float64
__device__ __forceinline__ double obs_stored(int type, double x) {
    if (type == OBS_F32) return (double)(float)x;
    if (type == OBS_BF16) return (double)bf16_to_f32(f32_to_bf16((float)x));
    return x;
}
// One action element, widened to float64 (exact for float32, so decode_order sees the same value a float64 caller passes)
__device__ __forceinline__ double load_action(const void* __restrict__ p, int64_t k, bool f32) {
    return f32 ? (double)reinterpret_cast<const float*>(p)[k] : reinterpret_cast<const double*>(p)[k];
}

// Reduced-precision observations: the table entry rounded on the host (float32: (float)tab[v] == np.float32(obs64); bfloat16:
// that float32 rounded to nearest even) — one 4- or 2-byte load and no F2F in the kernel (conversions run at a fraction of the
// FP64 rate; 7 per lane made the float32 step of config 2 SLOWER than the float64 one although it writes 112 fewer bytes per env)
template <typename T>
__device__ __forceinline__ T scaled_lp(const T* __restrict__ tabrow_lp, int TL, int which, int v) {
#ifdef IMX_DEBUG_BOUNDS
    if ((unsigned)v >= (unsigned)TL) __trap();
#endif
    return __ldg(tabrow_lp + which * TL + (int)min((unsigned)v, (unsigned)(TL - 1)));
}
// Row of the reduced-precision table for node i (null for float64 observations or without tables).
#define OBS_TABROW_LP(A, i, TL)                                                                                          \
    (!KHAS(tab) ? (const void*)nullptr                                                                                   \
     : KF(obs_type) == OBS_F32 ? (const void*)((A).tabf + (size_t)(i) * 4 * (TL))                                        \
     : KF(obs_type) == OBS_BF16 ? (const void*)((A).tabh + (size_t)(i) * 4 * (TL)) : (const void*)nullptr)

// The single writer of an observation element.  `row` addresses the agent's vector in the output element type.
#define OBS_PUT(row, k, v)                                                                                               \
    do {                                                                                                                 \
        if (KF(obs_type) == OBS_BF16) reinterpret_cast<uint16_t*>(row)[k] = f32_to_bf16((float)(v));                     \
        else if (KF(obs_type) == OBS_F32) reinterpret_cast<float*>(row)[k] = (float)(v);                                  \
        else reinterpret_cast<double*>(row)[k] = (v);                                                                    \
    } while (0)

// A rescaled element (scaled() above) and a raw integer element: for reduced-precision rows the host-rounded table / the
// int -> float conversion give the bits of the float32 (then bfloat16) rounding of the float64 value directly
// ((float)(double)i == (float)i for every int).
#define OBS_PUT_SCALED(row, k, CHECKED_, tabrow, tabrow_lp, TL, which, v, vmax, a, bma)                                  \
    do {                                                                                                                 \
        if (KF(obs_type) != OBS_F64 && KHAS(tab) && (!(CHECKED_) || (unsigned)(v) < (unsigned)(TL))) {                     \
            if (KF(obs_type) == OBS_BF16)                                                                                \
                reinterpret_cast<uint16_t*>(row)[k] = scaled_lp(reinterpret_cast<const uint16_t*>(tabrow_lp), TL, which, v); \
            else reinterpret_cast<float*>(row)[k] = scaled_lp(reinterpret_cast<const float*>(tabrow_lp), TL, which, v);  \
        } else OBS_PUT(row, k, scaled<CHECKED_>(KHAS(tab), tabrow, TL, which, v, vmax, a, bma));                          \
    } while (0)
#define OBS_PUT_INT(row, k, v)                                                                                           \
    do {                                                                                                                 \
        if (KF(obs_type) == OBS_BF16) reinterpret_cast<uint16_t*>(row)[k] = f32_to_bf16((float)(v));                     \
        else if (KF(obs_type) == OBS_F32) reinterpret_cast<float*>(row)[k] = (float)(v);                                  \
        else reinterpret_cast<double*>(row)[k] = (double)(v);                                                            \
    } while (0)

// profit = p*ship - c*order - h*|inv' - target| - bc*backlog'           MAIM_env.py:421-424
__device__ __forceinline__ double profit_of(double p, double c, double h, double bc, double target,
                                            int ship, int order, int inv_new, int backlog_new) {
    double r = __dsub_rn(__dmul_rn(p, (double)ship), __dmul_rn(c, (double)order));
    r = __dsub_rn(r, __dmul_rn(h, fabs(__dsub_rn((double)inv_new, target))));
    return __dsub_rn(r, __dmul_rn(bc, (double)backlog_new));
}

// ------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11), hand-rolled: counter-based, so a draw is a pure
// function of (seed, global env, index, period, episode) and independent of the sharding.
// ------------------------------------------------------------------------------------
struct Philox4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ void philox_mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
    const uint64_t p = (uint64_t)a * (uint64_t)b;
    hi = (uint32_t)(p >> 32);
    lo = (uint32_t)p;
}

__host__ __device__ __forceinline__ Philox4 philox4x32_10(Philox4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0, lo0, hi1, lo1;
        philox_mulhilo(0xD2511F53u, c.x, hi0, lo0);
        philox_mulhilo(0xCD9E8D57u, c.z, hi1, lo1);
        Philox4 n;
        n.x = hi1 ^ c.y ^ k0;
        n.y = lo1;
        n.z = hi0 ^ c.w ^ k1;
        n.w = lo0;
        c = n;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c;
}

enum : uint32_t { PHILOX_TAG_DEMAND = 0u, PHILOX_TAG_DELAY = 1u, PHILOX_TAG_DEMAND_NOISE = 2u };

// counter = (env_lo, env_hi, tag<<28 | idx<<16 | t, episode_lo), key = (seed_lo, seed_hi ^ episode_hi)
__host__ __device__ __forceinline__ Philox4 philox_draw(uint64_t seed, uint64_t env_global, uint32_t tag,
                                                        uint32_t idx, uint32_t t, uint64_t episode) {
    Philox4 c;
    c.x = (uint32_t)env_global;
    c.y = (uint32_t)(env_global >> 32);
    c.z = (tag << 28) | ((idx & 0xFFFu) << 16) | (t & 0xFFFFu);
    c.w = (uint32_t)episode;
    return philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32) ^ (uint32_t)(episode >> 32));
}

// 53-bit uniform in [0, 1) from two 32-bit words
__host__ __device__ __forceinline__ double u53(uint32_t hi, uint32_t lo) {
    const uint64_t bits = ((uint64_t)(hi >> 5) << 26) | (uint64_t)(lo >> 6);
    return (double)bits * (1.0 / 9007199254740992.0);
}

// Demand generator description (uniform kernel argument).
struct DemandGen {
    int32_t dist;                 // imx_demand_dist
    int32_t low, high;            // uniform integers in [low, high)
    int32_t cdf_len;              // Poisson: entries in cdf[]
    const double* __restrict__ cdf;       // Poisson CDF table, cdf[k] = P(X <= k); inversion: smallest k with u < cdf[k]
    const uint16_t* __restrict__ guide;   // cutpoint table: guide[g] = smallest k with cdf[k] > g / 256
    uint64_t seed;
    uint64_t episode;
    int64_t env_offset;
    double noise_thr;             // noisy demand (MAIM_div_env.py:287-295): 0 = off
};

// One uniform -> one demand.  Poisson by CDF inversion started from the cutpoint table (the scan
// from guide[floor(256 u)] reaches the same k as a search from 0, usually in 0-1 steps).
__device__ __forceinline__ int demand_from_uniform(const DemandGen& g, double u) {
    if (g.dist == IMX_DIST_UNIFORM) {
        const int k = g.low + (int)(u * (double)(g.high - g.low));
        return k < g.high ? k : g.high - 1;
    }
    int k = (int)__ldg(g.guide + (int)(u * 256.0));
    while (u >= __ldg(g.cdf + k)) ++k;          // the last table entry is a sentinel > 1
    return k;
}

// Noisy demand, MAIM_div_env.py:287-295 / IM_div_env.py: two uniforms per (retailer, period); "double" is
// applied before "zero", so a period that draws both ends at 0.  Own Philox tag, counter = the period.
__device__ __forceinline__ int demand_noise(const DemandGen& g, int64_t n_local, int r, int t, int d) {
    const Philox4 v = philox_draw(g.seed, (uint64_t)(g.env_offset + n_local), PHILOX_TAG_DEMAND_NOISE, (uint32_t)r, (uint32_t)t, g.episode);
    if (u53(v.x, v.y) <= g.noise_thr) d = 2 * d;
    if (u53(v.z, v.w) <= g.noise_thr) d = 0;
    return d;
}

// One Philox call serves TWO consecutive periods of one (env, retailer) row: the counter carries
// t >> 1, words (x, y) make the uniform of the even period and (z, w) of the odd one.
__device__ __forceinline__ void draw_demand_pair(const DemandGen& g, int64_t n_local, int r, int t_even, int& d0, int& d1) {
    const Philox4 v = philox_draw(g.seed, (uint64_t)(g.env_offset + n_local), PHILOX_TAG_DEMAND, (uint32_t)r,
                                  (uint32_t)(t_even >> 1), g.episode);
    d0 = demand_from_uniform(g, u53(v.x, v.y));
    d1 = demand_from_uniform(g, u53(v.z, v.w));
    if (KNOISY_DEMAND(g)) {                // a literal in the specialised build: the second Philox call must not bloat the rollout loop
        d0 = demand_noise(g, n_local, r, t_even, d0);
        d1 = demand_noise(g, n_local, r, t_even + 1, d1);
    }
}
__device__ __forceinline__ int draw_demand(const DemandGen& g, int64_t n_local, int r, int t) {
    int d0, d1;
    draw_demand_pair(g, n_local, r, t & ~1, d0, d1);
    return (t & 1) ? d1 : d0;
}

__device__ __forceinline__ bool draw_delay(uint64_t seed, int64_t env_global, int i, int t, uint64_t episode, double thr) {
    const Philox4 v = philox_draw(seed, (uint64_t)env_global, PHILOX_TAG_DELAY, (uint32_t)i, (uint32_t)t, episode);
    return u53(v.x, v.y) <= thr;
}

// ------------------------------------------------------------------------------------
// TMA bulk copy shared -> global (SASS: UBLKCP).  One elected lane issues it for a whole warp's
// contiguous observation tile, so the global write needs no per-lane store instructions.
// ------------------------------------------------------------------------------------
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void bulk_store_s2g(void* gdst, const void* ssrc, uint32_t bytes) {
    const uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(s), "r"(bytes)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// wait until the bulk engine has finished READING shared memory (the tile may then be overwritten)
__device__ __forceinline__ void bulk_wait_read_all() {
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// streaming global accesses: state and I/O are touched once per launch
__device__ __forceinline__ int ld_stream(const int32_t* p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream(int32_t* p, int v) { __stcs(p, v); }

}  // namespace imx
