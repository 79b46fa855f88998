// imx_api.cu — C ABI (include/imx_b200.h) over the sm_100a kernels: handle management, config
// validation and derivation, kernel dispatch.  No torch, no CPU fallback: every entry point
// either launches CUDA work or returns an error.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <new>
#include <vector>

#include <nvtx3/nvToolsExt.h>       // header-only; a no-op unless a profiler injects itself (SURVEY section 5: ranges around reset / step / rollout)

#include "imx_reset.cuh"
#include "imx_step_tma.cuh"
#include "imx_rollout.cuh"
#include "imx_step_pipe.cuh"
#include "imx_rollout_et.cuh"
#include "imx_kernels.cuh"
#include "imx_stats.cuh"
#include "imx_jit.cuh"
#include "imx_cc.cuh"
#include "imx_eval.cuh"

using namespace imx;

// --------------------------------------------------------------------------------------
// errors
// --------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define IMX_CUDA(call)                                                                             \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) return fail(-2, "%s failed: %s", #call, cudaGetErrorString(e__));   \
    } while (0)
#define IMX_CHECK_LAUNCH(name)                                                                     \
    do {                                                                                           \
        cudaError_t e__ = cudaGetLastError();                                                      \
        if (e__ != cudaSuccess) return fail(-3, "launch of %s failed: %s", name, cudaGetErrorString(e__)); \
        g_launches.fetch_add(1, std::memory_order_relaxed);                                        \
    } while (0)

// NVTX range of one entry point (domain "imx_b200"): shows up as reset / step / rollout spans on an nsys or ncu timeline.
struct NvtxRange {
    static nvtxDomainHandle_t domain() {
        static nvtxDomainHandle_t d = nvtxDomainCreateA("imx_b200");
        return d;
    }
    explicit NvtxRange(const char* name) { nvtxDomainRangePushEx(domain(), attr(name)); }
    ~NvtxRange() { nvtxDomainRangePop(domain()); }
    static const nvtxEventAttributes_t* attr(const char* name) {
        static thread_local nvtxEventAttributes_t a;
        memset(&a, 0, sizeof(a));
        a.version = NVTX_VERSION;
        a.size = NVTX_EVENT_ATTRIB_STRUCT_SIZE;
        a.messageType = NVTX_MESSAGE_TYPE_ASCII;
        a.message.ascii = name;
        return &a;
    }
};
#define IMX_NVTX(name) NvtxRange nvtx_range__(name)

extern "C" const char* imx_last_error(void) { return g_err; }
extern "C" int imx_abi_version(void) { return IMX_ABI_VERSION; }
extern "C" int imx_config_size(void) { return (int)sizeof(imx_config); }
extern "C" int64_t imx_launch_count(void) { return g_launches.load(); }

// --------------------------------------------------------------------------------------
// handle
// --------------------------------------------------------------------------------------
typedef void (*reset_fn_t)(const StepArgs, const ResetArgs, int);

struct imx_env {
    imx_config cfg;
    bool div, multi;
    int m, T, P, D, O, L, NB, R, maxc;
    int demand_max[IMX_MAX_NODES];
    int depth[IMX_MAX_NODES], parent[IMX_MAX_NODES], child_slot[IMX_MAX_NODES];
    int retailers[IMX_MAX_NODES], retailer_idx[IMX_MAX_NODES];
    double sell[IMX_MAX_NODES], buy[IMX_MAX_NODES];
    bool need_hd, need_ho, write_hd, has_carry;
    int S;                               // int32 state words per env
    int64_t N;
    // device memory
    NodeParams* d_nodes = nullptr;
    int32_t* d_state = nullptr;          // one block holding every state field
    size_t state_bytes = 0;
    void* field_ptr[IMX_F_COUNT] = {};
    int64_t field_cnt[IMX_F_COUNT] = {};
    int32_t* d_err = nullptr;
    int32_t* d_demand_T = nullptr;
    uint8_t* d_mask_T = nullptr;
    double* d_cdf = nullptr;
    uint16_t* d_guide = nullptr;         // cutpoint table of the Poisson inversion
    int cdf_len = 0;
    double* d_stats_partial = nullptr;   // [max(2 + 2m, 2(4 + m))][STATS_BLOCKS] scratch of imx_return_stats / imx_eval_stats
    double* d_dfo_rewards = nullptr;     // [T][N] scratch of the dfo objective (allocated on first use / imx_prepare)
    double* d_tab = nullptr;             // [m][4][TL] rescale tables
    int TL = 0;
    // host-call staging (allocated on first use)
    cudaStream_t hstream = nullptr;
    double *d_act_h = nullptr, *d_obs_h = nullptr, *d_rew_h = nullptr;   // (sized for float64; a float32 handle uses the first half)
    int32_t* d_dem_h = nullptr;
    uint8_t* d_mask_h = nullptr;
    // episode bookkeeping
    int t = 0;
    int noisy_now = 0;
    uint64_t episode = 0;
    // kernels
    step_fn_t step_fn = nullptr;
    tma_fn_t tma_fn = nullptr;
    tma_fn_t tma_many_fn = nullptr;      // the same kernel instantiated with the multi-period loop (imx_step_many)
    TileLayout tile = {};                // ahead-of-time kernels: tile width = m rounded up to a power of two
    TileLayout tile_jit = {};            // runtime-specialised kernels: tile width = m (dense lane packing)
    int step_path = 0;                   // 0 auto, 1 direct only, 2 TMA wherever legal (IMX_STEP_PATH)
    int host_zero_copy = 1;              // imx_step_host addresses pinned host buffers directly (IMX_HOST_ZERO_COPY=0: staged copies)
    int step_dense = 0;                  // experimental: m-wide tiles in the specialised step kernel (IMX_STEP_DENSE=1)
    int tma_threads = 256;               // CTA size of the TMA kernel (IMX_TMA_THREADS: 64, 128 or 256)
    int use_pdl = 1;                     // chain step launches with programmatic dependent launch (IMX_PDL=0 disables)
    int fuse_periods = 1;                // imx_step_many advances all its periods in one launch (IMX_FUSE_PERIODS=0: K plain launches)
    int l2_hints = 0;                    // L2 eviction priorities on the pipelined kernel's bulk copies (IMX_L2_HINTS; default: see select_kernels)
    int step_et = 0;                     // the specialised STEP kernels use the env-per-thread period (IMX_STEP_ET; default: divergent networks, m <= 8)
    int rollout_et = 0;                  // the specialised ROLLOUT kernel is the env-per-thread one (imx_rollout_et.cuh; IMX_ROLLOUT_ET, default m <= 8)
    int jit_threads = 128;               // CTA size (compute threads) of the specialised TMA kernels: tma_threads, or the env-per-thread group size
    int pipe_mode = 0;                   // persistent pipelined step kernel: 0 auto, 1 always, -1 never (IMX_PIPE)
    int pipe_stages = 0;                 // ring depth of the pipelined kernel (IMX_PIPE_STAGES; 0 = measured default)
    int pipe_ctas = 0;                   // resident CTAs per SM of the pipelined kernel (IMX_PIPE_CTAS; 0 = derived)
    int sm_count = 148;
    int jit_policy = 0;                  // 0 auto (large batches), 1 always, -1 never (IMX_JIT)
    int jit_state = 0;                   // 0 not tried, 1 specialised kernels loaded, -1 unavailable
    const imxjit::Kernels* jit = nullptr;
    const imxjit::Kernels* jit_noobs = nullptr;   // specialised without the observation output
    int jit_noobs_state = 0;
    const imxjit::Kernels* jit_cc = nullptr;      // specialised with the centralised-critic rows emitted by the step (imx_step_cc)
    int jit_cc_state = 0;
    TileLayout tile_cc = {};             // tile_jit + the [E][m][W] critic-row region
    void* d_obs_scratch = nullptr;       // [N][m][O] observations of the unfused imx_step_cc / imx_replay_episode when the caller passes none
    const imxjit::Kernels* jit_ep = nullptr;        // the one-launch episode kernel (imx_replay_episode) with observations ...
    const imxjit::Kernels* jit_ep_noobs = nullptr;  // ... and without
    int jit_ep_state = 0, jit_ep_noobs_state = 0;
    double* d_ep_rewards = nullptr;      // [T][N](m) rewards of the unfused imx_replay_episode when the caller passes none
    double* d_ep_profit = nullptr;       // [N][m] one period's profits (unfused imx_replay_episode with evaluation accumulators)
    double* d_ep_ret = nullptr;          // [N](m) returns of imx_replay_episode when only the statistics are wanted
    double* d_ep_stats = nullptr;        // [3 + 2m] statistics of the unfused imx_replay_episode when only the returns are wanted
    int last_variant = 0;                // 0 AOT direct, 1 AOT TMA, 2 runtime-specialised TMA, 3 pipelined, 4 one-launch episode
    reset_fn_t reset_fn = nullptr;
    rollout_fn_t rollout_fn = nullptr;
    int step_grid_cap = 0, rollout_grid_cap = 0;
    size_t step_smem = 0;
    int m_pad = 0;
};

// The per-handle I/O element types (imx_config.obs_f32 / io_flags): every size the host derives from them comes from here.
static int obs_type_of(const imx_config& c) { return (c.io_flags & IMX_IO_OBS_BF16) ? OBS_BF16 : c.obs_f32 ? OBS_F32 : OBS_F64; }
static int obs_elem_bytes(const imx_env* e) { return imx::obs_elem_bytes(obs_type_of(e->cfg)); }
static int act_elem_bytes(const imx_env* e) { return (e->cfg.io_flags & IMX_IO_ACTIONS_F32) ? 4 : 8; }
// bytes one step moves per env: state read + written, demand, actions, rewards, observations
static int64_t bytes_per_env(const imx_env* e) {
    return 8 * (int64_t)e->S + 4 * e->R + (int64_t)e->m * (act_elem_bytes(e) + 8 + e->O * obs_elem_bytes(e));
}

// --------------------------------------------------------------------------------------
// kernel dispatch tables: the template instantiations live in imx_kernels_inst.cu, one object per
// (tile width, network family), compiled in parallel by the build
// --------------------------------------------------------------------------------------
#define IMX_DECL_PICK(MP, DV) void imx_pick_kernels_##MP##_##DV(bool small, bool few, imx::KernelSet* ks);
IMX_DECL_PICK(2, 0) IMX_DECL_PICK(4, 0) IMX_DECL_PICK(8, 0) IMX_DECL_PICK(16, 0) IMX_DECL_PICK(32, 0)
IMX_DECL_PICK(4, 1) IMX_DECL_PICK(8, 1) IMX_DECL_PICK(16, 1) IMX_DECL_PICK(32, 1)
#undef IMX_DECL_PICK

static int m_pad_of(const imx_env* e);
static void pick_kernels(imx_env* e, int m_pad, bool div) {
    const bool small = (e->D <= 4 && e->P <= 1);
    const bool few = e->maxc <= 2;
    KernelSet ks;
    if (div) {
        if (m_pad == 4) imx_pick_kernels_4_1(small, few, &ks);
        else if (m_pad == 8) imx_pick_kernels_8_1(small, few, &ks);
        else if (m_pad == 16) imx_pick_kernels_16_1(small, few, &ks);
        else imx_pick_kernels_32_1(small, few, &ks);
    } else {
        if (m_pad == 2) imx_pick_kernels_2_0(small, few, &ks);
        else if (m_pad == 4) imx_pick_kernels_4_0(small, few, &ks);
        else if (m_pad == 8) imx_pick_kernels_8_0(small, few, &ks);
        else if (m_pad == 16) imx_pick_kernels_16_0(small, few, &ks);
        else imx_pick_kernels_32_0(small, few, &ks);
    }
    e->step_fn = ks.step_fn; e->tma_fn = ks.tma_fn; e->tma_many_fn = ks.tma_many_fn; e->rollout_fn = ks.rollout_fn;
    const int ot = obs_type_of(e->cfg);
    if (ot == OBS_BF16) e->reset_fn = small ? reset_kernel<4, 1, OBS_BF16> : reset_kernel<8, 8, OBS_BF16>;
    else if (ot == OBS_F32) e->reset_fn = small ? reset_kernel<4, 1, OBS_F32> : reset_kernel<8, 8, OBS_F32>;
    else e->reset_fn = small ? reset_kernel<4, 1, OBS_F64> : reset_kernel<8, 8, OBS_F64>;
    e->m_pad = m_pad;
}

// The dynamic-shared-memory limit is an attribute of the FUNCTION, shared by every handle that uses the same
// instantiation: only ever raise it (a handle with a smaller tile must not lower it under a live handle's launches).
static cudaError_t raise_dyn_smem_limit(const void* fn, size_t bytes) {
    cudaFuncAttributes fa;
    cudaError_t rc = cudaFuncGetAttributes(&fa, fn);
    if (rc != cudaSuccess) return rc;
    if ((size_t)fa.maxDynamicSharedSizeBytes >= bytes) return cudaSuccess;
    return cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

static int m_pad_of(const imx_env* e);

// CTA size of the TMA kernel.  128-thread CTAs de-synchronise the load / compute / store phases of neighbouring tiles and
// measured faster on every shipped config (profiles/r1_other_configs_1gpu.jsonl) except the 4-wide chain at
// multi-million-env batches, where the 256-thread tile is 2.5% ahead; 512-thread CTAs lose 25%
static int choose_tma_threads(const imx_env* e) {
    const char* tt = getenv("IMX_TMA_THREADS");
    // 4-wide serial chains in the pipelined regime (working set within ~1.5 x L2, see pipe_pays): 64-thread tiles of 16 envs with
    // 8 resident CTAs per SM measured 3 % ahead of 128-thread tiles (profiles/r2_pipe_sweep.txt); 256-thread tiles from 1 Mi envs
    const bool small4 = !e->div && m_pad_of(e) == 4 && e->N >= 1024 && bytes_per_env(e) * e->N <= ((int64_t)192 << 20);
    // (512 Ki envs of a 4-wide chain, pipelined with the L2 priorities: 256-thread tiles 35.7 us, 128-thread 38.1, 64-thread 38.9)
    const bool big4 = !e->div && m_pad_of(e) == 4 && e->N >= ((int64_t)1 << 19);
    const int dflt = small4 ? 64 : (big4 || (m_pad_of(e) <= 4 && e->N >= ((int64_t)1 << 20))) ? 256 : 128;
    const int v = tt ? atoi(tt) : dflt;
    return ((v == 64 || v == 128 || v == 256 || v == 512) && v >= 2 * m_pad_of(e)) ? v : 256;
}

static int m_pad_of(const imx_env* e) {
    const int m = e->m;
    if (e->div) return m <= 4 ? 4 : m <= 8 ? 8 : m <= 16 ? 16 : 32;
    return m <= 2 ? 2 : m <= 4 ? 4 : m <= 8 ? 8 : m <= 16 ? 16 : 32;
}

// shared-memory tile layout of the TMA kernel (regions 128-byte aligned); pure host arithmetic
static void compute_tile(const imx_env* e, TileLayout& L, int tile_width, bool with_cc = false, int E_fixed = 0) {
    const int m = e->m;
    // lanes = nodes: (warps per CTA) x (envs per warp); env-per-thread: one env per compute thread (E_fixed)
    const int E = E_fixed > 0 ? E_fixed : (e->tma_threads / 32) * (32 / tile_width);
    int off = 0;
    auto take = [&](int bytes) { const int o = off; off += (bytes + 127) & ~127; return o; };
    L.E = E;
    // the multi-period kernel's shared-reward scratch ([E][m] float64) lives in the action region: over the consumed float64 actions,
    // behind float32 ones (which other warps may still be reading when a lane stores its profit)
    const int act_region = E * m * (act_elem_bytes(e) == 4 ? 12 : 8);
    L.off_act = take(act_region);
    L.off_inv = take(E * m * 4);
    L.off_bl = take(E * m * 4);
    L.off_ou = take(E * m * 4);
    L.off_pipe = take(E * e->L * 4);
    L.off_hd = take(e->need_hd ? E * m * e->P * 4 : 0);
    L.off_ho = take(e->need_ho ? E * m * e->P * 4 : 0);
    L.off_carry = take(e->has_carry ? E * m * 4 : 0);
    L.off_bt = take(E * e->NB * 4);
    L.off_dem = take(e->R * E * 4);
    L.off_obs = take(E * m * e->O * obs_elem_bytes(e));
    L.off_rew = take(E * m * 8);
    L.off_cc = with_cc ? take(E * m * ((m - 1) * (1 + e->O) + e->O) * obs_elem_bytes(e)) : 0;
    L.total = off;
    // multi-period launches double-buffer the per-period inputs; the extra regions sit behind the
    // single-period layout so that a plain step launches the same kernel with `total` bytes only
    L.off_act2 = take(act_region);
    L.off_dem2 = take(e->R * E * 4);
    L.total2 = off;
}

// -D options and template instantiations of the runtime-specialised build (imx_jit.cuh)
// Ring depth of the pipelined kernel for a given tile layout.  Measured shapes (profiles/r2_pipe_sweep.txt, r2_step_et_sweep.txt):
// four stages for the lane-mapped tiles, two for the env-per-thread tiles (their 32-env tiles are 2-3 x larger: a deeper ring
// costs resident CTAs); the critic-row variant shortens its ring until four CTAs fit on an SM.
static int pipe_stages_for(const imx_env* e, const TileLayout& L) {
    const bool is_cc = (&L == &e->tile_cc);
    int s = e->pipe_stages > 0 ? e->pipe_stages : ((e->step_et && !is_cc) ? 2 : 4);
    while (s > 2 && ((int64_t)s * L.total > 200 * 1024 || (is_cc && (227 * 1024) / ((int64_t)s * L.total + 1024) < 4))) --s;
    return s;
}

// episode != 0: the module holds the one-launch episode kernel only (imx_replay_episode)
static void jit_spec(const imx_env* e, int TL, imxjit::Spec& sp, int has_obs = 1, int has_cc = 0, int episode = 0) {
    std::vector<std::string>& defs = sp.defines;
    const imx_config& c = e->cfg;
    const bool always_std = (c.kind == IMX_KIND_MAIM_DIV);
    const int std_state = always_std ? 1 : (c.standardise_state != 0);
    auto add = [&](const char* k, long long v) { defs.push_back(std::string("IMX_K_") + k + "=" + std::to_string(v)); };
    add("m", e->m); add("T", e->T); add("P", e->P); add("D", e->D); add("O", e->O); add("L", e->L); add("NB", e->NB);
    add("R", e->R); add("maxc", e->maxc); add("multi", e->multi); add("std_state", std_state);
    add("std_actions", always_std ? 1 : (c.standardise_actions != 0)); add("cap_backlog", always_std ? 1 : std_state);
    add("independent", c.independent != 0); add("share_network", (c.kind == IMX_KIND_MAIM_DIV && c.share_network) ? 1 : 0);
    add("td", c.time_dependency != 0); add("pd", c.prev_demand != 0); add("pa", c.prev_actions != 0);
    add("write_hd", e->write_hd); add("has_carry", e->has_carry); add("need_hd", e->need_hd);
    // noisy delays: a handle without the carry state never has them (literal 0); one with it decides per episode (reset(noisy=...)),
    // so the specialised kernels of such a handle read the flag from the argument block
    defs.push_back(e->has_carry ? "IMX_K_noisy=(A.noisy)" : "IMX_K_noisy=0");
    add("need_ho", e->need_ho); add("wd_mult1", e->multi ? 2 : 4); add("wd_mult", e->multi ? 1 : 2); add("TL", TL);
    add("noisy_demand", (e->div && c.noisy_demand_threshold > 0.0) ? 1 : 0); add("has_info", 0); add("has_obs", has_obs); add("has_tab", TL > 0);
    add("obs_type", obs_type_of(c)); add("act_f32", (c.io_flags & IMX_IO_ACTIONS_F32) ? 1 : 0);
    int ex = 0;
    const double fr = std::frexp(c.b - c.a, &ex);
    add("bma_pow2", (fr == 0.5 && ex > -1000 && ex < 1000) ? 1 : 0);
    add("m_pow2", ((e->m & (e->m - 1)) == 0) ? 1 : 0);
    const TileLayout& L = has_cc ? e->tile_cc : e->tile_jit;
    add("has_cc", has_cc);
    auto addt = [&](const char* k, long long v) { defs.push_back(std::string("IMX_KT_") + k + "=" + std::to_string(v)); };
    addt("E", L.E); addt("off_act", L.off_act); addt("off_inv", L.off_inv); addt("off_bl", L.off_bl); addt("off_ou", L.off_ou);
    addt("off_pipe", L.off_pipe); addt("off_hd", L.off_hd); addt("off_ho", L.off_ho); addt("off_carry", L.off_carry);
    addt("off_bt", L.off_bt); addt("off_dem", L.off_dem); addt("off_obs", L.off_obs); addt("off_rew", L.off_rew); addt("total", L.total);
    addt("off_act2", L.off_act2); addt("off_dem2", L.off_dem2); addt("total2", L.total2); addt("off_cc", L.off_cc);
    {   // L2 eviction priorities on the bulk copies (IMX_L2_HINTS=1: observation stream evict_first, state and rewards evict_last)
        if (e->l2_hints) defs.push_back("IMX_L2_HINTS=" + std::to_string(e->l2_hints));
    }
    {   // L2 prefetch of the action tiles ahead of griddepcontrol.wait (IMX_ACT_PREFETCH=0 switches it off for A/B runs)
        const char* ap = getenv("IMX_ACT_PREFETCH");
        if (ap && !strcmp(ap, "0")) defs.push_back("IMX_NO_ACT_PREFETCH=1");
    }
    {   // register bound of the plain step kernel, measured per family: the divergent kernels (natural 47) gain occupancy at 40
        // (div1 +5 %, div2 +1.5 %), the 2-wide chain is faster unconstrained (+8 % at 64), the others are best at their natural 32
        const char* sr = getenv("IMX_STEP_MAXNREG");
        const int bound = sr ? atoi(sr) : (e->step_et ? 0 : e->div ? 40 : (m_pad_of(e) == 2 ? 64 : 0));   // (the env-per-thread kernels spill at 40)
        if (bound > 0) defs.push_back("IMX_STEP_MAXNREG=" + std::to_string(bound));
    }
    {   // register bound of the rollout kernel.  Measured (profiles/r1_other_configs_1gpu.jsonl): the divergent kernel wants
        // ~90 registers and is latency-bound at 6 CTAs/SM — 72 buys occupancy (+6 %); the serial multi-agent kernel spills at
        // its natural 72 — 96 removes the spills (+3 %); the single-agent kernel is best left alone.  IMX_ROLLOUT_MAXNREG overrides.
        const char* rr = getenv("IMX_ROLLOUT_MAXNREG");
        const int bound = rr ? atoi(rr) : (e->div ? 72 : (e->multi ? 96 : 0));
        if (bound > 0) defs.push_back("IMX_ROLLOUT_MAXNREG=" + std::to_string(bound));
    }
    {   // register bound of the multi-period kernel (IMX_MANY_MAXNREG=0: none)
        const char* mr = getenv("IMX_MANY_MAXNREG");
        const int maxnreg = mr ? atoi(mr) : 0;             // 0: the per-config default in imx_step_tma.cuh
        if (maxnreg > 0) defs.push_back("IMX_MANY_MAXNREG=" + std::to_string(maxnreg));
    }
    defs.push_back("IMX_TMA_THREADS=" + std::to_string((has_cc && e->step_et) ? e->tma_threads : e->jit_threads));
    // the device translation unit checks its view of the argument blocks against this host build (imx_jit.cuh)
    defs.push_back("IMX_HOST_SIZEOF_STEPARGS=" + std::to_string(sizeof(StepArgs)));
    defs.push_back("IMX_HOST_SIZEOF_TILELAYOUT=" + std::to_string(sizeof(TileLayout)));
    defs.push_back("IMX_HOST_SIZEOF_ROLLOUTARGS=" + std::to_string(sizeof(RolloutArgs)));
    defs.push_back("IMX_HOST_SIZEOF_EPISODEARGS=" + std::to_string(sizeof(EpisodeArgs)));
    const int mp = e->step_dense ? e->m : m_pad_of(e);     // step kernel: power-of-two tile width (see select_kernels)
    const int pmax = (e->need_hd || e->need_ho) ? e->P : 1;
    const int maxc = e->maxc > 1 ? e->maxc : 1;
    const std::string dv = e->div ? "true" : "false";
    const std::string targs = "<" + std::to_string(mp) + ", " + std::to_string(e->D) + ", " + std::to_string(pmax) + ", " +
                              std::to_string(e->div ? maxc : 1) + ", " + dv + ">";
    sp.name[0] = "imx::step_kernel_tma" + targs;
    sp.name[1] = "imx::step_kernel_tma_many" + targs;
    const bool step_et = e->step_et && !has_cc;            // (the critic-row variant keeps the lane mapping and its tile geometry)
    if (e->rollout_et || step_et) {
        // env-per-thread kernels: the network as compile-time integer lists
        auto list = [&](const char* k, auto get) {
            std::string v;
            for (int i = 0; i < e->m; ++i) v += (i ? "," : "") + std::to_string((long long)get(i));
            defs.push_back(std::string("IMX_L_") + k + "=" + v);
        };
        if (e->rollout_et) defs.push_back("IMX_ET=1");
        if (step_et) {
            defs.push_back("IMX_STEP_ET=1");
            auto bits = [&](const char* k, auto get) {
                std::string v;
                for (int i = 0; i < e->m; ++i) {
                    const double d = get(i);
                    unsigned long long u;
                    memcpy(&u, &d, 8);
                    char buf[32];
                    snprintf(buf, sizeof(buf), "0x%016llxull", u);
                    v += (i ? "," : "") + std::string(buf);
                }
                defs.push_back(std::string("IMX_L_") + k + "=" + v);
            };
            bits("p_bits", [&](int i) { return e->sell[i]; });
            bits("c_bits", [&](int i) { return e->buy[i]; });
            bits("h_bits", [&](int i) { return c.stock_cost[i]; });
            bits("bc_bits", [&](int i) { return c.backlog_cost[i]; });
            bits("target_bits", [&](int i) { return c.inv_target[i]; });
        }
        list("inv_max", [&](int i) { return c.inv_max[i]; });
        list("order_max", [&](int i) { return c.order_max[i]; });
        list("demand_max", [&](int i) { return e->demand_max[i]; });
        list("delay", [&](int i) { return c.delay[i]; });
        list("init_inv", [&](int i) { return c.inv_init[i]; });
        list("nchild", [&](int i) { return e->div ? c.num_children[i] : 0; });
        list("retailer_idx", [&](int i) { return e->retailer_idx[i]; });
        {
            std::string po, bo, ch;
            int p_off = 0, b_off = 0;
            for (int i = 0; i < e->m; ++i) {
                po += (i ? "," : "") + std::to_string(p_off);
                p_off += c.delay[i];
                const bool split = e->div && c.num_children[i] > 1;
                bo += (i ? "," : "") + std::to_string(split ? b_off : -1);
                if (split) b_off += c.num_children[i];
                for (int k = 0; k < maxc; ++k)
                    ch += ((i || k) ? "," : "") + std::to_string((e->div && k < c.num_children[i]) ? c.children[i][k] : -1);
            }
            defs.push_back("IMX_L_pipe_off=" + po);
            defs.push_back("IMX_L_bt_off=" + bo);
            defs.push_back("IMX_L_children=" + ch);
        }
    }
    if (e->rollout_et) {
        sp.name[2] = "imx::rollout_kernel_et<" + std::to_string(e->m) + ", " + std::to_string(e->D) + ", " + std::to_string(maxc) + ", " + dv + ">";
    } else
        sp.name[2] = "imx::rollout_kernel<" + std::to_string(e->m) + ", " + std::to_string(e->D) + ", " + std::to_string(e->div ? maxc : 1) +
                     ", " + dv + ">";
    sp.name[3] = "";
    if (has_cc) { sp.name[1] = ""; sp.name[2] = ""; }      // the critic rows ride on the single-period kernels only
    if (e->pipe_mode >= 0 && (int64_t)pipe_stages_for(e, L) * L.total <= 200 * 1024) {
        defs.push_back("IMX_PIPE_STAGES=" + std::to_string(pipe_stages_for(e, L)));
        const char* pr = getenv("IMX_PIPE_MAXNREG");
        if (pr && atoi(pr) > 0) defs.push_back("IMX_PIPE_MAXNREG=" + std::to_string(atoi(pr)));
        sp.name[3] = "imx::step_kernel_pipe" + targs;
    }
    sp.name[4] = "";
    if (episode) {
        for (int k = 0; k < 4; ++k) sp.name[k] = "";
        sp.name[4] = "imx::step_kernel_tma_episode" + targs;
    }
}

static void jit_smem(const imx_env* e, int smem[imxjit::N_KERNELS]) {
    smem[0] = e->tile_jit.total;
    smem[1] = e->tile_jit.total2 <= 200 * 1024 ? e->tile_jit.total2 : e->tile_jit.total;
    smem[2] = 0;
    smem[3] = pipe_stages_for(e, e->tile_jit) * e->tile_jit.total;
    smem[4] = 0;
}

// Loads the specialised kernels for this handle (large batches, or IMX_JIT=1).  Called from imx_create() /
// imx_prepare(); a later call only happens for handles whose policy changed, and never under stream capture.
static void ensure_jit(imx_env* e) {
    if (e->jit_state != 0) return;
    e->jit_state = -1;
    if (e->jit_policy < 0 || !e->tma_fn) return;
    if (e->jit_policy == 0 && e->N < 1024) return;        // below ~1k envs a step is launch latency either way; the compile (1-2 s) is not worth it
    if (e->tile_jit.total > 200 * 1024) return;
    imxjit::Spec sp;
    jit_spec(e, e->TL, sp);
    int smem[imxjit::N_KERNELS];
    jit_smem(e, smem);
    e->jit = imxjit::get(sp, smem, e->cfg.device);
    if (e->jit) e->jit_state = 1;
}

// The same kernels specialised WITHOUT an observation output (step / step_many with obs = NULL: scoring a stored plan
// needs rewards only — the observation build and 60 % of the bytes fold away).  Compiled by imx_prepare(IMX_PREPARE_NOOBS)
// or on first use outside stream capture.
static void ensure_jit_noobs(imx_env* e) {
    if (e->jit_noobs_state != 0) return;
    e->jit_noobs_state = -1;
    ensure_jit(e);
    if (e->jit_state != 1) return;
    imxjit::Spec sp;
    jit_spec(e, e->TL, sp, 0);
    int smem[imxjit::N_KERNELS];
    jit_smem(e, smem);
    e->jit_noobs = imxjit::get(sp, smem, e->cfg.device);
    if (e->jit_noobs) e->jit_noobs_state = 1;
}

// ... and WITH the centralised-critic rows (imx_step_cc).  Compiled by imx_prepare(IMX_PREPARE_CC) or on first use outside capture.
static void ensure_jit_cc(imx_env* e) {
    if (e->jit_cc_state != 0) return;
    e->jit_cc_state = -1;
    ensure_jit(e);
    if (e->jit_state != 1 || !e->multi || e->tile_cc.total > 200 * 1024) return;
    imxjit::Spec sp;
    jit_spec(e, e->TL, sp, 1, 1);
    int smem[imxjit::N_KERNELS] = {e->tile_cc.total, 0, 0, pipe_stages_for(e, e->tile_cc) * e->tile_cc.total};
    if (smem[3] > 200 * 1024) smem[3] = 0;
    e->jit_cc = imxjit::get(sp, smem, e->cfg.device);
    if (e->jit_cc) e->jit_cc_state = 1;
}

// Shared-memory layout of the episode kernel: tile_jit's multi-period layout, then the episode regions of EpisodeArgs that the
// call needs (the returns and the accumulators adjacent: the kernel zeroes [off_ret, off_prof) in one loop) — a launch reserves
// no bytes it does not use, since resident CTAs per SM bound this latency-bound loop.  Returns the total bytes.
static int64_t episode_layout(const imx_env* e, EpisodeArgs& EA, bool ret = true, bool eval = true) {
    const int64_t E = e->tile_jit.E, cols = e->multi ? e->m : 1;
    int64_t off = e->tile_jit.total2;
    auto take = [&](int64_t bytes) { const int64_t o = off; off += (bytes + 127) & ~(int64_t)127; return (int32_t)(o < (1 << 30) ? o : 0); };
    EA.off_edem = take(E * e->R * e->T * 4);
    EA.off_ret = take(ret ? E * cols * 8 : 0);
    EA.off_eval = take(eval ? E * (EVAL_FIXED + e->m) * 8 : 0);
    EA.off_prof = take(eval ? E * e->m * 8 : 0);
    EA.total = (int32_t)(off < (1 << 30) ? off : 0);
    return off;
}

// The episode kernel, with (obs) or without observations.  Compiled by imx_prepare(IMX_PREPARE_EPISODE) or on first use
// outside stream capture; unavailable where the specialised kernels are (small batches) or the layout exceeds 200 KB.
static void ensure_jit_episode(imx_env* e, bool obs) {
    int& st = obs ? e->jit_ep_state : e->jit_ep_noobs_state;
    if (st != 0) return;
    st = -1;
    ensure_jit(e);
    EpisodeArgs EA;
    if (e->jit_state != 1 || episode_layout(e, EA) > 200 * 1024) return;
    imxjit::Spec sp;
    jit_spec(e, e->TL, sp, obs ? 1 : 0, 0, 1);
    const int smem[imxjit::N_KERNELS] = {0, 0, 0, 0, EA.total};
    const imxjit::Kernels* k = imxjit::get(sp, smem, e->cfg.device);
    (obs ? e->jit_ep : e->jit_ep_noobs) = k;
    if (k) st = 1;
}

static bool stream_is_capturing(cudaStream_t s) {
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(s, &st) != cudaSuccess) { cudaGetLastError(); return false; }
    return st != cudaStreamCaptureStatusNone;
}

// see the comment at the call in select_kernels(); l2_bytes <= 0: the B200's 126 MB (imx_jit_compile_check runs without a device)
static int decide_l2_hints(const imx_env* e, int l2_bytes) {
    if (l2_bytes <= 0) l2_bytes = 126 << 20;
    const int64_t per_env = bytes_per_env(e);
    const int64_t state_bytes = 4 * (int64_t)e->S * e->N;
    const char* lh = getenv("IMX_L2_HINTS");
    if (lh && !strcmp(lh, "1")) return 1;
    if (lh && !strcmp(lh, "2")) return 2;                  // outputs only (measurement switch)
    if (lh && !strcmp(lh, "0")) return 0;
    // below the window: outputs only (2) — the step itself is unchanged (everything is L2-resident), but the step rewards are
    // still in L2 when imx_episode_stats reads them back after 30 periods of observation traffic (config 2 episode 205.2 -> 202.1 us,
    // 32 768 envs 143.2 -> 140.3 us; profiles/r2_l2_hints_small_ab.txt)
    if (per_env * e->N <= (int64_t)l2_bytes / 2) return 2;
    return state_bytes <= (int64_t)l2_bytes * 5 / 8 ? 1 : 0;
}

static int select_kernels(imx_env* e) {
    const int m = e->m;
    pick_kernels(e, m_pad_of(e), e->div);
    const int epw = 32 / e->m_pad;
    const int tile_bytes = (epw * m * e->O * obs_elem_bytes(e) + 15) & ~15;
    e->step_smem = (size_t)(STEP_THREADS / 32) * tile_bytes;
    IMX_CUDA(raise_dyn_smem_limit((const void*)e->step_fn, e->step_smem));
    int dev_sms = 0, occ = 0;
    IMX_CUDA(cudaDeviceGetAttribute(&dev_sms, cudaDevAttrMultiProcessorCount, e->cfg.device));
    IMX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, (const void*)e->step_fn, STEP_THREADS, e->step_smem));
    if (occ < 1) return fail(-4, "step kernel does not fit on an SM (smem %zu B)", e->step_smem);
    e->step_grid_cap = dev_sms * occ;
    {
        e->tma_threads = choose_tma_threads(e);
        const char* dn = getenv("IMX_STEP_DENSE");
        e->step_dense = (dn && !strcmp(dn, "1")) ? 1 : 0;
    }
    compute_tile(e, e->tile, m_pad_of(e));
    // the specialised STEP kernel keeps the power-of-two tile: a dense m-wide tile makes the per-field byte
    // ranges (e.g. 40 envs x 6 nodes x 4 B = 960 B) straddle 128-byte lines, measured slower at 262144 envs;
    // the issue-bound ROLLOUT kernel is specialised with tile width = m (dense lane packing, +21% on div2)
    {
        // env-per-thread rollout (imx_rollout_et.cuh): networks up to 8 nodes, lead times up to 4 (registers); IMX_ROLLOUT_ET=0 disables
        const char* re = getenv("IMX_ROLLOUT_ET");
        e->rollout_et = (re && !strcmp(re, "0")) ? 0 : (e->m <= 8 && e->D <= 4);
        // env-per-thread STEP kernels: divergent networks up to 8 nodes (their lane-mapped kernels are issue-bound); IMX_STEP_ET=0/1
        const char* se = getenv("IMX_STEP_ET");
        const bool et_ok = e->m <= 8 && e->D <= 4 && e->P <= 2;
        // default: divergent networks whose node count is not a power of two (the lane mapping pads them: div2 runs 19 of 32 lanes);
        // div2 262 144 envs 34.9 -> 33.6 us, 1 Mi envs 129 -> 115 us; no gain on the 4-node div1 (profiles/r2_step_et_sweep.txt)
        const bool non_pow2 = (e->m & (e->m - 1)) != 0;
        e->step_et = (se && !strcmp(se, "0")) ? 0 : (se && !strcmp(se, "1")) ? et_ok : (et_ok && e->div && non_pow2);
        const char* st = getenv("IMX_STEP_ET_THREADS");
        const int et_threads = (st && (atoi(st) == 32 || atoi(st) == 64 || atoi(st) == 128)) ? atoi(st) : 32;
        e->jit_threads = e->step_et ? et_threads : e->tma_threads;
    }
    compute_tile(e, e->tile_jit, e->step_dense ? e->m : m_pad_of(e), false, e->step_et ? e->jit_threads : 0);
    compute_tile(e, e->tile_cc, e->step_dense ? e->m : m_pad_of(e), true);
    if (e->tile.total <= 200 * 1024) {
        IMX_CUDA(raise_dyn_smem_limit((const void*)e->tma_fn, (size_t)e->tile.total));
        if (e->tile.total2 <= 200 * 1024)
            IMX_CUDA(raise_dyn_smem_limit((const void*)e->tma_many_fn, (size_t)e->tile.total2));
    }
    else
        e->tma_fn = nullptr;
    {
        const char* pth = getenv("IMX_STEP_PATH");
        e->step_path = (pth && !strcmp(pth, "direct")) ? 1 : (pth && !strcmp(pth, "tma")) ? 2 : 0;
        const char* zc = getenv("IMX_HOST_ZERO_COPY");
        e->host_zero_copy = (zc && !strcmp(zc, "0")) ? 0 : 1;
        const char* pd = getenv("IMX_PDL");
        e->use_pdl = (pd && !strcmp(pd, "0")) ? 0 : 1;
        const char* fu = getenv("IMX_FUSE_PERIODS");
        e->fuse_periods = (fu && !strcmp(fu, "0")) ? 0 : 1;
        const char* jp = getenv("IMX_JIT");
        e->jit_policy = (jp && !strcmp(jp, "1")) ? 1 : (jp && !strcmp(jp, "0")) ? -1 : 0;
        const char* pm = getenv("IMX_PIPE");
        e->pipe_mode = (pm && !strcmp(pm, "1")) ? 1 : (pm && !strcmp(pm, "0")) ? -1 : 0;
        const char* ps = getenv("IMX_PIPE_STAGES");
        e->pipe_stages = ps ? atoi(ps) : 0;                 // 0: the measured default of pipe_stages_for()
        if (e->pipe_stages < 2 || e->pipe_stages > 8) e->pipe_stages = 0;
        const char* pc = getenv("IMX_PIPE_CTAS");
        e->pipe_ctas = pc ? atoi(pc) : 0;
        e->sm_count = dev_sms;
        // L2 eviction priorities (observation stream evict_first, state + rewards evict_last): they pay exactly where a launch
        // streams more than about half of L2 while the state itself would still fit — the write-once stream then no longer
        // pushes the state out between two periods (config 2 at 262 144 envs 20.7 -> 16.6 us = 1.15 of the HBM copy peak, div2
        // 33.4 -> 27.1 us, 8-stage 49.2 -> 43.0 us); below that everything is L2-resident anyway (-1 %), above it the state does
        // not fit and the priorities only disturb the replacement (-2 .. -4 %).  profiles/r2_l2_hints_ab.txt
        int l2_bytes = 0;
        cudaDeviceGetAttribute(&l2_bytes, cudaDevAttrL2CacheSize, e->cfg.device);
        e->l2_hints = decide_l2_hints(e, l2_bytes);
    }
    IMX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, (const void*)e->rollout_fn, ROLLOUT_THREADS, 0));
    if (occ < 1) return fail(-4, "rollout kernel does not fit on an SM");
    e->rollout_grid_cap = dev_sms * occ;
    return 0;
}

// --------------------------------------------------------------------------------------
// config validation + derivation (host mirror of the reference constructors)
// --------------------------------------------------------------------------------------
static int derive(imx_env* e) {
    const imx_config& c = e->cfg;
    if (c.kind < IMX_KIND_IM || c.kind > IMX_KIND_MAIM_DIV) return fail(-1, "unknown kind %d", c.kind);
    e->div = (c.kind == IMX_KIND_IM_DIV || c.kind == IMX_KIND_MAIM_DIV);
    e->multi = (c.kind == IMX_KIND_MAIM || c.kind == IMX_KIND_MAIM_DIV);
    const int m = e->m = c.num_nodes;
    if (m < 1 || m > IMX_MAX_NODES) return fail(-1, "num_nodes %d outside [1, %d]", m, IMX_MAX_NODES);
    if (e->div && m < 2) return fail(-1, "a divergent network needs at least 2 nodes");
    e->T = c.num_periods;
    if (e->T < 1 || e->T > 65535) return fail(-1, "num_periods %d outside [1, 65535]", e->T);
    e->P = c.prev_length;
    const bool uses_hist = c.prev_demand || c.prev_actions;
    if (uses_hist && (e->P < 1 || e->P > IMX_MAX_HIST)) return fail(-1, "prev_length %d outside [1, %d]", e->P, IMX_MAX_HIST);
    if (!uses_hist) e->P = (e->P < 1) ? 1 : (e->P > IMX_MAX_HIST ? IMX_MAX_HIST : e->P);
    e->N = c.num_envs;
    if (e->N < 1) return fail(-1, "num_envs must be >= 1");
    if (!(c.b != c.a)) return fail(-1, "rescale interval needs a != b");
    if (e->multi && !c.time_dependency && c.prev_actions && !c.prev_demand)
        return fail(-5, "Not Implemented");   // MAIM_env.py:135-136, MAIM_div_env.py:164-165
    if (c.io_flags & ~(IMX_IO_OBS_BF16 | IMX_IO_ACTIONS_F32))
        return fail(-1, "io_flags 0x%x has unknown bits (known: IMX_IO_OBS_BF16 = 1, IMX_IO_ACTIONS_F32 = 2)", (unsigned)c.io_flags);
    if ((c.io_flags & IMX_IO_OBS_BF16) && c.obs_f32)
        return fail(-1, "obs_f32 and IMX_IO_OBS_BF16 both set: choose one observation element type");

    e->D = 0;
    e->L = 0;
    for (int i = 0; i < m; ++i) {
        if (c.delay[i] < 1 || c.delay[i] > IMX_MAX_DELAY)
            return fail(-1, "delay[%d] = %d outside [1, %d]", i, c.delay[i], IMX_MAX_DELAY);
        if (c.inv_max[i] < 1) return fail(-1, "inv_max[%d] must be >= 1", i);
        if (c.order_max[i] < 1) return fail(-1, "order_max[%d] must be >= 1", i);
        if (c.inv_init[i] < 0) return fail(-1, "init_inv[%d] must be >= 0", i);
        if (c.inv_max[i] > (1 << 28) || c.order_max[i] > (1 << 28)) return fail(-1, "capacities above 2^28 are not supported");
        e->D = c.delay[i] > e->D ? c.delay[i] : e->D;
        e->L += c.delay[i];
    }

    for (int i = 0; i < m; ++i) { e->parent[i] = -1; e->child_slot[i] = -1; e->retailer_idx[i] = -1; e->depth[i] = 0; }
    e->maxc = 0;
    e->NB = 0;
    e->R = 0;
    if (e->div) {
        for (int p = 0; p < m; ++p) {
            const int nc = c.num_children[p];
            if (nc < 0 || nc > IMX_MAX_CHILDREN) return fail(-1, "node %d has %d children (max %d)", p, nc, IMX_MAX_CHILDREN);
            e->maxc = nc > e->maxc ? nc : e->maxc;
            for (int k = 0; k < nc; ++k) {
                const int ch = c.children[p][k];
                if (ch == p) return fail(-1, "node %d lists itself as a child (utils.py:87-92 lets this through; the reference then never terminates its depth walk)", p);
                if (ch < p || ch >= m)   // utils.py:87-92
                    return fail(-1, "Downstream node cannot have a smaller index number than upstream node (%d -> %d)", p, ch);
                if (e->parent[ch] != -1) return fail(-1, "node %d has more than one upstream node", ch);
                e->parent[ch] = p;
                e->child_slot[ch] = k;
            }
        }
        for (int i = 1; i < m; ++i) {
            if (e->parent[i] < 0) return fail(-1, "node %d is not connected to node 0", i);
            e->depth[i] = e->depth[e->parent[i]] + 1;          // parents have smaller indices
        }
        for (int i = 0; i < m; ++i) {
            if (c.num_children[i] == 0) { e->retailer_idx[i] = e->R; e->retailers[e->R++] = i; }
            e->sell[i] = (double)(e->depth[i] + 2);            // MAIM_div_env.py:55-61
            e->buy[i] = (double)(e->depth[i] + 1);
            int64_t s = 0;                                     // MAIM_div_env.py:91-99
            for (int k = 0; k < c.num_children[i]; ++k) s += c.order_max[c.children[i][k]];
            if (s > INT32_MAX)
                return fail(-1, "demand_max[%d] = %lld (the sum of its children's order_max) exceeds INT32_MAX: the int32 state "
                                "cannot hold it", i, (long long)s);
            e->demand_max[i] = s > c.inv_max[i] ? (int)s : c.inv_max[i];
        }
        if (c.order_max[0] > c.inv_max[0]) return fail(-1, "order_max[0] must not exceed inv_max[0]");   // MAIM_div_env.py:235
    } else {
        e->R = 1;
        e->retailers[0] = 0;
        e->retailer_idx[0] = 0;
        for (int i = 0; i < m; ++i) {
            if (!(c.price[i] > c.price[i + 1])) return fail(-1, "price must be strictly decreasing (MAIM_env.py:167-168)");
            e->sell[i] = c.price[i];
            e->buy[i] = c.price[i + 1];
            e->demand_max[i] = c.inv_max[i];
        }
        if (c.order_max[m - 1] > c.inv_max[m - 1]) return fail(-1, "order_max of the last stage must not exceed its inv_max (MAIM_env.py:171)");
    }

    const bool std_state = (c.kind == IMX_KIND_MAIM_DIV) ? true : (c.standardise_state != 0);
    // Domain of the int32 state (the reference's integers are unbounded).  A node's demand in one period is at most dmax_i:
    // the clipped customer demand of a retailer, a serial stage's downstream order, a split node's children's orders.  An
    // uncapped backlog (standardise_state = 0 on IM, IM_div and MAIM) grows by at most dmax_i a period, and so does a split node's
    // per-child ledger (IMX_F_BACKLOG_TO, never capped, negative entries bounded by earlier positive ones): both stay below
    // T * dmax_i, which must fit int32.  Every other int32 quantity is bounded by a capacity (<= 2^28) or by these.
    for (int i = 0; i < m; ++i) {
        int64_t dmax = (e->retailer_idx[i] >= 0) ? c.inv_max[i] : e->div ? 0 : c.order_max[i - 1];
        if (e->div)
            for (int k = 0; k < c.num_children[i]; ++k) dmax += c.order_max[c.children[i][k]];
        const int64_t bound = (int64_t)e->T * dmax;
        if (bound > INT32_MAX && !std_state)
            return fail(-1, "num_periods * the largest per-period demand of node %d = %lld exceeds INT32_MAX: its uncapped backlog "
                            "(standardise_state = 0) could wrap the int32 state", i, (long long)bound);
        if (bound > INT32_MAX && e->div && c.num_children[i] > 1)
            return fail(-1, "num_periods * the largest per-period demand of node %d = %lld exceeds INT32_MAX: its per-child backlog "
                            "ledger could wrap the int32 state", i, (long long)bound);
        // The noisy-delay carry (IMX_F_CARRY) holds every arrival of a run of delayed periods, and acquisition adds it to the
        // inventory.  A node receives no more over the episode than it orders (T * order_max_i): its supplier ships at most
        // the backlog plus demand it owes, or the factory fills the order itself.  A divergent child can receive up to twice
        // that, since the split subtracts what it ships from the parent's ledger twice when it drains a backlog, and the
        // ledger may then go negative by as much as it was positive.
        if (c.noisy_delay) {
            const int64_t arrivals = (int64_t)e->T * c.order_max[i] * ((e->div && i > 0) ? 2 : 1);
            if (arrivals + c.inv_max[i] > INT32_MAX)
                return fail(-1, "with noisy delays, inv_max[%d] + the most node %d can receive over num_periods (%lld) exceeds "
                                "INT32_MAX: goods held back over consecutive delayed periods could wrap the int32 state", i, i,
                                (long long)arrivals);
        }
    }
    // quirk 2: MAIM kinds in mode (td=F, pd=T, pa=F) never write the demand-history slots
    e->write_hd = !(e->multi && c.prev_demand && !c.prev_actions && !c.time_dependency);
    e->need_hd = c.prev_demand && e->write_hd && !(e->multi && !std_state);
    e->need_ho = c.prev_actions && !(e->multi && !std_state);
    e->has_carry = c.noisy_delay != 0;
    e->O = 3 + (c.prev_demand ? e->P : 0) + (c.prev_actions ? e->P : 0) + (c.time_dependency ? e->D : 0)
         + ((c.kind == IMX_KIND_MAIM_DIV && c.share_network) ? 1 : 0);
    e->NB = 0;
    if (e->div)
        for (int i = 0; i < m; ++i)
            if (c.num_children[i] > 1) e->NB += c.num_children[i];
    e->S = 3 * m + e->L + (e->need_hd ? m * e->P : 0) + (e->need_ho ? m * e->P : 0) + (e->has_carry ? m : 0) + e->NB;

    if (c.demand_dist == IMX_DIST_POISSON && !(c.mu > 0.0 && c.mu <= 1000.0)) return fail(-1, "mu must be in (0, 1000]");
    if (c.demand_dist == IMX_DIST_UNIFORM && !(c.uniform_low < c.uniform_high))
        return fail(-1, "Lower bound cannot be larger than upper bound");    // MAIM_env.py:215-216
    if (c.demand_dist < IMX_DIST_REPLAY_ONLY || c.demand_dist > IMX_DIST_UNIFORM)
        return fail(-1, "Unrecognised, Distribution Not Implemented");        // MAIM_env.py:219
    return 0;
}

static void launch_reset_kernel(imx_env* e, double* obs_dev, cudaStream_t s, const int32_t* demand_in = nullptr);

static void fill_args(const imx_env* e, StepArgs& A) {
    const imx_config& c = e->cfg;
    memset(&A, 0, sizeof(A));
    A.N = e->N; A.m = e->m; A.T = e->T; A.P = e->P; A.D = e->D; A.O = e->O; A.L = e->L; A.NB = e->NB; A.R = e->R;
    A.t = e->t;
    A.maxc = e->maxc;
    A.multi = e->multi;
    const bool always_std = (c.kind == IMX_KIND_MAIM_DIV);    // quirk 9
    A.std_state = always_std ? 1 : (c.standardise_state != 0);
    A.std_actions = always_std ? 1 : (c.standardise_actions != 0);
    A.cap_backlog = always_std ? 1 : A.std_state;
    A.independent = c.independent != 0;
    A.share_network = (c.kind == IMX_KIND_MAIM_DIV && c.share_network);
    A.td = c.time_dependency != 0; A.pd = c.prev_demand != 0; A.pa = c.prev_actions != 0;
    A.write_hd = e->write_hd;
    A.noisy = e->noisy_now;
    A.has_carry = e->has_carry;
    A.need_hd = e->need_hd; A.need_ho = e->need_ho;
    A.obs_type = obs_type_of(c);
    A.act_f32 = (c.io_flags & IMX_IO_ACTIONS_F32) ? 1 : 0;
    // watchdog thresholds: MAIM_div 2*dm, dm, dm, dm (:504,526,560,574); IM_div 4*dm, 2*dm, 2*dm, 2*dm (:424,449,483,497)
    A.wd_mult1 = e->multi ? 2 : 4;
    A.wd_mult = e->multi ? 1 : 2;
    A.a = c.a; A.b = c.b; A.bma = c.b - c.a;
    {
        int ex = 0;
        const double fr = std::frexp(A.bma, &ex);          // power of two <=> mantissa exactly 0.5
        A.inv_bma = (fr == 0.5 && ex > -1000 && ex < 1000) ? 1.0 / A.bma : 0.0;
        A.inv_m = 1.0 / (double)e->m;
        A.m_pow2 = ((e->m & (e->m - 1)) == 0) ? 1 : 0;
    }
    A.TL = e->TL;
    A.tab = e->d_tab;
    A.tabf = e->d_tab ? reinterpret_cast<const float*>(e->d_tab + (size_t)e->m * 4 * e->TL) : nullptr;   // float32 copy behind the float64 table
    A.tabh = e->d_tab ? reinterpret_cast<const uint16_t*>(A.tabf + (size_t)e->m * 4 * e->TL) : nullptr; // bfloat16 copy behind that
    A.nodes = e->d_nodes;
    A.inv = (int32_t*)e->field_ptr[IMX_F_INV];
    A.backlog = (int32_t*)e->field_ptr[IMX_F_BACKLOG];
    A.order_u = (int32_t*)e->field_ptr[IMX_F_ORDER_U];
    A.pipe = (int32_t*)e->field_ptr[IMX_F_PIPE];
    A.hist_d = (int32_t*)e->field_ptr[IMX_F_HIST_D];
    A.hist_o = (int32_t*)e->field_ptr[IMX_F_HIST_O];
    A.carry = (int32_t*)e->field_ptr[IMX_F_CARRY];
    A.bt = (int32_t*)e->field_ptr[IMX_F_BACKLOG_TO];
    A.err = e->d_err;
    A.demand_T = e->d_demand_T;
    A.mask_T = e->d_mask_T;
}

// Exact rescale tables: tab[i][k][v] = a + (v*(b-a))/max_k(i), evaluated with the same three IEEE
// double operations as MAIM_env.py:505 (this translation unit is compiled with -ffp-contract=off
// semantics: product, quotient and sum are separate roundings).  Row k: 0 scale inv_max, 1 order_max,
// 2 demand_max, 3 MAIM_div pipeline min(v, 2*inv_max)/(2*inv_max).
static std::vector<double> build_tables(const imx_env* e, int* TL_out) {
    const imx_config& c = e->cfg;
    int maxv = 1;
    for (int i = 0; i < e->m; ++i) {
        maxv = c.inv_max[i] > maxv ? c.inv_max[i] : maxv;
        maxv = c.order_max[i] > maxv ? c.order_max[i] : maxv;
        maxv = e->demand_max[i] > maxv ? e->demand_max[i] : maxv;
    }
    const int64_t TL = 2 * (int64_t)maxv + IMX_MAX_CHILDREN + 8 + 1;   // covers every reachable value (DESIGN.md §tables)
    if (TL * 4 * e->m * (int64_t)sizeof(double) > (int64_t)8 << 20) { *TL_out = 0; return {}; }
    std::vector<double> tab((size_t)e->m * 4 * TL);
    const volatile double a = c.a, bma = c.b - c.a;
    for (int i = 0; i < e->m; ++i) {
        const double mx[4] = {(double)c.inv_max[i], (double)c.order_max[i], (double)e->demand_max[i], 2.0 * (double)c.inv_max[i]};
        for (int k = 0; k < 4; ++k)
            for (int64_t v = 0; v < TL; ++v) {
                double x = (double)v;
                if (k == 3 && v > 2 * (int64_t)c.inv_max[i]) x = 2.0 * (double)c.inv_max[i];
                volatile double prod = x * bma;
                volatile double quot = prod / mx[k];
                tab[((size_t)i * 4 + k) * TL + v] = a + quot;
            }
    }
    *TL_out = (int)TL;
    return tab;
}

// float32 -> bfloat16 bits, round to nearest even: the rounding of torch's float -> bfloat16 conversion (c10::BFloat16)
static uint16_t round_bf16(float f) {
    if (std::isnan(f)) return 0x7FC0;
    uint32_t u;
    memcpy(&u, &f, 4);
    u += 0x7FFFu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
extern "C" int imx_round_bf16(const float* in, uint16_t* out, int64_t n) {
    if ((!in || !out) && n > 0) return fail(-1, "null argument");
    for (int64_t k = 0; k < n; ++k) out[k] = round_bf16(in[k]);
    return 0;
}

static std::vector<double> poisson_cdf(double mu) {
    // cdf[k] = sum_{j<=k} exp(j*log(mu) - lgamma(j+1) - mu); stop once the tail is below 2^-53
    std::vector<double> cdf;
    double acc = 0.0;
    for (int k = 0; k < 8192; ++k) {
        acc += std::exp(k * std::log(mu) - std::lgamma(k + 1.0) - mu);
        cdf.push_back(acc);
        if (k > mu && 1.0 - acc < 1.2e-16) break;
    }
    cdf.back() = 2.0;   // sentinel: the search always terminates inside the table
    return cdf;
}

extern "C" int imx_create(const imx_config* cfg, imx_env** out) {
    if (!cfg || !out) return fail(-1, "null argument");
    *out = nullptr;
    imx_env* e = new (std::nothrow) imx_env();
    if (!e) return fail(-1, "out of host memory");
    e->cfg = *cfg;
    int rc = derive(e);
    if (rc) { delete e; return rc; }
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0) {
        delete e;
        return fail(-2, "no CUDA device available (%s) — this library has no CPU fallback", cudaGetErrorString(ce));
    }
    if (cfg->device < 0 || cfg->device >= ndev) { delete e; return fail(-1, "device %d out of range", cfg->device); }
#define IMX_CREATE_CUDA(call)                                                                      \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            fail(-2, "%s failed: %s", #call, cudaGetErrorString(e__));                              \
            imx_destroy(e);                                                                        \
            return -2;                                                                             \
        }                                                                                          \
    } while (0)
    IMX_CREATE_CUDA(cudaSetDevice(cfg->device));
    rc = select_kernels(e);
    if (rc) { imx_destroy(e); return rc; }

    const int m = e->m;
    const int64_t N = e->N;
    // node table
    NodeParams h_nodes[IMX_MAX_NODES];
    memset(h_nodes, 0, sizeof(h_nodes));
    int pipe_off = 0, bt_off = 0;
    for (int i = 0; i < m; ++i) {
        NodeParams& q = h_nodes[i];
        q.inv_max = cfg->inv_max[i]; q.order_max = cfg->order_max[i]; q.demand_max = e->demand_max[i];
        q.delay = cfg->delay[i]; q.pipe_off = pipe_off; pipe_off += cfg->delay[i];
        q.init_inv = cfg->inv_init[i];
        q.parent = e->parent[i]; q.child_slot = e->child_slot[i];
        q.nchild = e->div ? cfg->num_children[i] : 0;
        q.bt_off = -1;
        if (e->div && cfg->num_children[i] > 1) { q.bt_off = bt_off; bt_off += cfg->num_children[i]; }
        q.retailer_idx = e->retailer_idx[i];
        q.parent_nchild = (e->div && e->parent[i] >= 0) ? cfg->num_children[e->parent[i]] : 0;
        q.p = e->sell[i]; q.c = e->buy[i]; q.h = cfg->stock_cost[i]; q.bc = cfg->backlog_cost[i]; q.target = cfg->inv_target[i];
        q.child_lo = q.child_hi = 0xFFFFFFFFu;
        if (e->div)
            for (int k = 0; k < cfg->num_children[i]; ++k) {
                uint32_t& w = (k < 4) ? q.child_lo : q.child_hi;
                w = (w & ~(0xFFu << ((k & 3) * 8))) | ((uint32_t)cfg->children[i][k] << ((k & 3) * 8));
            }
    }
    IMX_CREATE_CUDA(cudaMalloc(&e->d_nodes, sizeof(h_nodes)));
    IMX_CREATE_CUDA(cudaMemcpy(e->d_nodes, h_nodes, sizeof(h_nodes), cudaMemcpyHostToDevice));

    // state block: fields back to back, each 256-byte aligned
    const int64_t cnt[IMX_F_COUNT] = {
        N * m, N * m, N * m, N * e->L,
        e->need_hd ? N * m * e->P : 0, e->need_ho ? N * m * e->P : 0,
        e->has_carry ? N * m : 0, N * e->NB, 0, 0, 0};
    size_t off[IMX_F_COUNT] = {};
    size_t total = 0;
    for (int f = 0; f <= IMX_F_BACKLOG_TO; ++f) {
        off[f] = total;
        total += ((size_t)cnt[f] * sizeof(int32_t) + 255) & ~(size_t)255;
    }
    e->state_bytes = total;
    IMX_CREATE_CUDA(cudaMalloc(&e->d_state, total ? total : 256));
    for (int f = 0; f <= IMX_F_BACKLOG_TO; ++f) {
        e->field_cnt[f] = cnt[f];
        e->field_ptr[f] = cnt[f] ? (void*)((char*)e->d_state + off[f]) : nullptr;
    }
    IMX_CREATE_CUDA(cudaMalloc(&e->d_err, (size_t)N * sizeof(int32_t)));
    e->field_ptr[IMX_F_ERROR] = e->d_err;
    e->field_cnt[IMX_F_ERROR] = N;
    const size_t dem_bytes = (size_t)e->T * e->R * N * sizeof(int32_t);
    IMX_CREATE_CUDA(cudaMalloc(&e->d_demand_T, dem_bytes));
    e->field_ptr[IMX_F_DEMAND] = e->d_demand_T;
    e->field_cnt[IMX_F_DEMAND] = (int64_t)e->T * e->R * N;
    if (e->has_carry) {
        IMX_CREATE_CUDA(cudaMalloc(&e->d_mask_T, (size_t)e->T * N * m));
        IMX_CREATE_CUDA(cudaMemset(e->d_mask_T, 0, (size_t)e->T * N * m));
        e->field_ptr[IMX_F_DELAY_MASK] = e->d_mask_T;
        e->field_cnt[IMX_F_DELAY_MASK] = (int64_t)e->T * N * m;
    }
    if (cfg->demand_dist == IMX_DIST_POISSON) {
        std::vector<double> cdf = poisson_cdf(cfg->mu);
        e->cdf_len = (int)cdf.size();
        IMX_CREATE_CUDA(cudaMalloc(&e->d_cdf, cdf.size() * sizeof(double)));
        IMX_CREATE_CUDA(cudaMemcpy(e->d_cdf, cdf.data(), cdf.size() * sizeof(double), cudaMemcpyHostToDevice));
        uint16_t guide[256];
        int k = 0;
        for (int g = 0; g < 256; ++g) {                       // smallest k with cdf[k] > g/256
            while (!(cdf[k] > (double)g / 256.0)) ++k;
            guide[g] = (uint16_t)k;
        }
        IMX_CREATE_CUDA(cudaMalloc(&e->d_guide, sizeof(guide)));
        IMX_CREATE_CUDA(cudaMemcpy(e->d_guide, guide, sizeof(guide), cudaMemcpyHostToDevice));
    }
    {
        std::vector<double> tab = build_tables(e, &e->TL);
        if (e->TL > 0) {
            // [m][4][TL] float64, then the same entries rounded to float32 (what an obs_f32 kernel stores: np.float32(obs64)), then
            // those rounded to bfloat16 (what an IMX_IO_OBS_BF16 kernel stores: torch's float64 -> bfloat16, which rounds through float32)
            std::vector<float> tabf(tab.size());
            std::vector<uint16_t> tabh(tab.size());
            for (size_t k = 0; k < tab.size(); ++k) { tabf[k] = (float)tab[k]; tabh[k] = round_bf16(tabf[k]); }
            IMX_CREATE_CUDA(cudaMalloc(&e->d_tab, tab.size() * (sizeof(double) + sizeof(float) + sizeof(uint16_t))));
            IMX_CREATE_CUDA(cudaMemcpy(e->d_tab, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice));
            IMX_CREATE_CUDA(cudaMemcpy(e->d_tab + tab.size(), tabf.data(), tab.size() * sizeof(float), cudaMemcpyHostToDevice));
            IMX_CREATE_CUDA(cudaMemcpy(reinterpret_cast<float*>(e->d_tab + tab.size()) + tab.size(), tabh.data(), tab.size() * sizeof(uint16_t),
                                       cudaMemcpyHostToDevice));
        }
    }
    {   // partial sums of the two-stage statistics: [statistic][slice] (imx_stats.cuh) or [2 x column][STATS_BLOCKS] (imx_eval.cuh)
        const int cols = e->multi ? m : 1;
        const int64_t nslices = (N + stats_envs_per_block(cols) - 1) / stats_envs_per_block(cols);
        const size_t a = (size_t)(2 + 2 * cols) * (size_t)nslices, b = (size_t)(2 * EVAL_FIXED + 2 + 2 * IMX_MAX_NODES) * STATS_BLOCKS;
        IMX_CREATE_CUDA(cudaMalloc(&e->d_stats_partial, (a > b ? a : b) * sizeof(double)));
    }
    // reset state with an all-zero demand trace (the reference constructors end with self.reset())
    IMX_CREATE_CUDA(cudaMemset(e->d_demand_T, 0, dem_bytes));
    {
        launch_reset_kernel(e, nullptr, nullptr);
        cudaError_t le = cudaGetLastError();
        if (le != cudaSuccess) { fail(-3, "reset launch failed: %s", cudaGetErrorString(le)); imx_destroy(e); return -3; }
        g_launches.fetch_add(1);
        IMX_CREATE_CUDA(cudaDeviceSynchronize());
    }
#undef IMX_CREATE_CUDA
    ensure_jit(e);            // compile / load the specialised kernels now: no later call compiles on the step path
    *out = e;
    return 0;
}

extern "C" int imx_destroy(imx_env* e) {
    if (!e) return 0;
    cudaSetDevice(e->cfg.device);
    if (e->hstream) { cudaStreamSynchronize(e->hstream); cudaStreamDestroy(e->hstream); }
    cudaFree(e->d_nodes); cudaFree(e->d_state); cudaFree(e->d_err);
    cudaFree(e->d_demand_T); cudaFree(e->d_mask_T); cudaFree(e->d_cdf); cudaFree(e->d_guide); cudaFree(e->d_tab); cudaFree(e->d_stats_partial);
    cudaFree(e->d_dfo_rewards); cudaFree(e->d_obs_scratch);
    cudaFree(e->d_ep_rewards); cudaFree(e->d_ep_profit); cudaFree(e->d_ep_ret); cudaFree(e->d_ep_stats);
    cudaFree(e->d_act_h); cudaFree(e->d_obs_h); cudaFree(e->d_rew_h); cudaFree(e->d_dem_h); cudaFree(e->d_mask_h);
    delete e;
    return 0;
}

// --------------------------------------------------------------------------------------
// getters
// --------------------------------------------------------------------------------------
extern "C" int imx_obs_len(const imx_env* e) { return e ? e->O : fail(-1, "null env"); }
extern "C" int imx_state_words(const imx_env* e) { return e ? e->S : fail(-1, "null env"); }
extern "C" int imx_num_retailers(const imx_env* e) { return e ? e->R : fail(-1, "null env"); }
extern "C" int imx_pipe_words(const imx_env* e) { return e ? e->L : fail(-1, "null env"); }
extern "C" int imx_ledger_words(const imx_env* e) { return e ? e->NB : fail(-1, "null env"); }
extern "C" int imx_retailers(const imx_env* e, int32_t* out) {
    if (!e || !out) return fail(-1, "null argument");
    for (int k = 0; k < e->R; ++k) out[k] = e->retailers[k];
    return 0;
}
extern "C" int imx_demand_max(const imx_env* e, int32_t* out) {
    if (!e || !out) return fail(-1, "null argument");
    for (int i = 0; i < e->m; ++i) out[i] = e->demand_max[i];
    return 0;
}
extern "C" int imx_node_price(const imx_env* e, double* sell, double* buy) {
    if (!e || !sell || !buy) return fail(-1, "null argument");
    for (int i = 0; i < e->m; ++i) { sell[i] = e->sell[i]; buy[i] = e->buy[i]; }
    return 0;
}
extern "C" int imx_state_field(imx_env* e, int field, void** dev_ptr, int64_t* count) {
    if (!e || !dev_ptr || !count) return fail(-1, "null argument");
    if (field < 0 || field >= IMX_F_COUNT) return fail(-1, "unknown field %d", field);
    *dev_ptr = e->field_ptr[field];
    *count = e->field_cnt[field];
    return 0;
}
extern "C" int imx_period(const imx_env* e) { return e ? e->t : fail(-1, "null env"); }
extern "C" int imx_set_period(imx_env* e, int t) {
    if (!e) return fail(-1, "null env");
    if (t < 0 || t > e->T) return fail(-1, "period %d outside [0, %d]", t, e->T);
    e->t = t;
    return 0;
}

// --------------------------------------------------------------------------------------
// reset / step
// --------------------------------------------------------------------------------------
// launches the reset fill kernel (state zero + inv init + optional t = 0 observation)
static void launch_reset_kernel(imx_env* e, double* obs_dev, cudaStream_t s, const int32_t* demand_in) {
    StepArgs A;
    fill_args(e, A);
    A.obs = obs_dev;
    ResetArgs Z;
    Z.zero_base = e->d_state;
    Z.zero_words = (int64_t)(e->state_bytes / sizeof(int32_t));
    Z.err = e->d_err;
    Z.demand_in = demand_in;                               // replayed trace [N][R][T]: transposed to [T][R][N] by the same launch
    Z.demand_T = e->d_demand_T;
    Z.R = e->R; Z.T = e->T;
    const int64_t work = (obs_dev ? e->N * e->m * e->O : 0) > Z.zero_words / 4 ? e->N * e->m * e->O : Z.zero_words / 4;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->cfg.device);
    int64_t blocks = (work + 255) / 256;
    if (blocks > (int64_t)sms * 8) blocks = (int64_t)sms * 8;
    if (blocks < 1) blocks = 1;
    const size_t smem = (size_t)e->m * e->O * sizeof(double) + (size_t)e->m * sizeof(int32_t);   // template sized for float64
    // a programmatic dependent of whatever is in front of it on the stream (the kernel starts with griddepcontrol.wait)
    cudaLaunchConfig_t lc;
    memset(&lc, 0, sizeof(lc));
    lc.gridDim = dim3((unsigned)blocks); lc.blockDim = dim3(256); lc.dynamicSmemBytes = smem; lc.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = at;
    lc.numAttrs = e->use_pdl ? 1 : 0;
    cudaLaunchKernelEx(&lc, e->reset_fn, A, Z, e->div ? 1 : 0);
}

static DemandGen make_gen(const imx_env* e, uint64_t episode) {
    DemandGen g;
    g.dist = e->cfg.demand_dist; g.low = e->cfg.uniform_low; g.high = e->cfg.uniform_high;
    g.cdf_len = e->cdf_len; g.cdf = e->d_cdf; g.guide = e->d_guide; g.seed = e->cfg.seed; g.episode = episode; g.env_offset = e->cfg.env_offset;
    g.noise_thr = e->div ? e->cfg.noisy_demand_threshold : 0.0;
    return g;
}

extern "C" int imx_reset(imx_env* e, const int32_t* demand_dev, const uint8_t* delay_mask_dev, int noisy,
                         uint64_t episode, void* obs_dev, void* stream) {
    IMX_NVTX("imx_reset");

    if (!e) return fail(-1, "null env");
    cudaStream_t s = (cudaStream_t)stream;
    IMX_CUDA(cudaSetDevice(e->cfg.device));
    if ((noisy || delay_mask_dev) && !e->has_carry) return fail(-1, "noisy delay requested but the env was created with noisy_delay = 0");
    if (!demand_dev && e->cfg.demand_dist == IMX_DIST_REPLAY_ONLY)
        return fail(-1, "reset() without a demand trace needs demand_dist poisson or uniform");
    const int64_t N = e->N;
    const unsigned gb = (unsigned)((N * e->R + 255) / 256);
    if (!demand_dev) {                                       // (a replayed trace is transposed by the reset kernel itself)
        demand_generate_kernel<<<gb, 256, 0, s>>>(e->d_demand_T, N, e->R, e->T, make_gen(e, episode));
        IMX_CHECK_LAUNCH("demand_generate_kernel");
    }
    e->noisy_now = (noisy || delay_mask_dev) ? 1 : 0;
    const int64_t cells = N * e->m;
    const unsigned cb = (unsigned)((cells + 255) / 256);
    if (e->noisy_now) {
        if (delay_mask_dev) {
            mask_transpose_kernel<<<cb, 256, 0, s>>>(delay_mask_dev, e->d_mask_T, N, e->m, e->T);
            IMX_CHECK_LAUNCH("mask_transpose_kernel");
        } else {
            mask_generate_kernel<<<cb, 256, 0, s>>>(e->d_mask_T, N, e->m, e->T, e->cfg.seed, e->cfg.env_offset, episode,
                                                    e->cfg.noisy_delay_threshold);
            IMX_CHECK_LAUNCH("mask_generate_kernel");
        }
    }
    e->t = 0;
    e->episode = episode;
    launch_reset_kernel(e, (double*)obs_dev, s, demand_dev);
    IMX_CHECK_LAUNCH("reset_kernel");
    return 0;
}

// auto policy, measured (profiles/r2_pipe_sweep.txt): the pipelined kernel wins at every batch size on the divergent
// networks (issue-bound kernels: +5-15 %) and on the serial chains while a launch's working set stays within ~1.5 x L2
// (one-wave regime: -3 % .. -20 % per launch; even with one tile per CTA its compute warps retire early, which lets the
// next dependent launch in sooner); for larger serial batches the one-tile-per-CTA kernel already runs at the HBM copy peak
// and the ring's smaller resident tile count costs 5-10 %.
static bool pipe_pays(const imx_env* e, int n_tiles) {
    (void)n_tiles;
    if (e->step_et) return bytes_per_env(e) * e->N <= ((int64_t)384 << 20);   // env-per-thread tiles: one-tile kernel from ~0.5 Mi envs (div2: 115 vs 124 us at 1 Mi)
    if (e->div) return true;
    if (e->l2_hints) return true;                          // the priorities live in the pipelined kernel (serial 4-stage at 512 Ki envs: 38.0 vs 41.8 us)
    return bytes_per_env(e) * e->N <= ((int64_t)192 << 20);
}
// CTAs launched per SM by the pipelined kernel (tiles are dealt round-robin over the grid).  Measured per family: 8 for the
// 64-thread tiles of 4-wide chains, 6 for 8-lane divergent tiles and for the env-per-thread tiles (more CTAs than fit at once:
// the late ones shorten everybody's tile list, which measured faster than a grid of exactly the resident CTAs), 4 otherwise.
static int pipe_ctas_for(const imx_env* e, const TileLayout& L) {
    const bool is_cc = (&L == &e->tile_cc);
    int want = 4;
    if (e->pipe_ctas > 0) want = e->pipe_ctas;
    else if (e->step_et && !is_cc) want = 6;
    else if (e->div) want = m_pad_of(e) <= 4 ? 4 : 6;
    else if (e->jit_threads == 64) want = 8;
    // never more than shared memory lets in (228 KB per SM, 1 KB reserved per CTA + the barriers): the tiles are assigned
    // statically, so CTAs that only become resident in a second wave would serialise the launch (float64 critic rows of the
    // 2-stage chain: 3 CTAs fit, a grid of 4 per SM took 11.0 us instead of 6)
    const int64_t per_cta = (int64_t)pipe_stages_for(e, L) * L.total + 1024 + 256;
    const int fit = (int)((228 * 1024) / per_cta);
    if (want > fit) want = fit;
    return want < 1 ? 1 : want;
}

// periods > 1 (imx_step_many): the TMA kernel advances that many periods in one launch with the tiles' state resident
// in shared memory; *done receives how many periods the call really advanced (1 when the fused form is not applicable:
// tail tiles, diagnostics, the direct path, a layout that does not fit).
struct CcOut { void* dev; int fill; double lo, hi; };
// The TMA kernels move a tile's actions, observations (and critic rows) as bulk copies, each of which must be a whole number of
// 16-byte units; with 4- and 2-byte elements that depends on E * m (* O).  Where it does not hold, the direct kernel serves.
static bool tile_io_whole16(const imx_env* e, const TileLayout& L, bool cc) {
    const int64_t cells = (int64_t)L.E * e->m;
    if ((cells * act_elem_bytes(e)) % 16 != 0 || (cells * e->O * obs_elem_bytes(e)) % 16 != 0) return false;
    return !cc || (cells * ((e->m - 1) * (1 + e->O) + e->O) * obs_elem_bytes(e)) % 16 == 0;
}
constexpr unsigned ET_THREADS_HOST = 128;     // = imx::ET_THREADS of the env-per-thread rollout (device-only constant)

static int launch_step(imx_env* e, const void* actions_dev, double* obs_dev, double* reward_dev,
                       const imx_info_out* info, cudaStream_t s, int periods = 1, int* done = nullptr, const CcOut* cc = nullptr,
                       bool* cc_fused = nullptr) {
    if (e->t >= e->T) return fail(-6, "step() past the end of the episode (period %d of %d)", e->t, e->T);
    StepArgs A;
    fill_args(e, A);
    const size_t cells_all = (size_t)e->N * e->m;
    A.periods = 1;
    A.act_stride = (int64_t)cells_all;
    A.obs_stride_bytes = (int64_t)(cells_all * e->O * obs_elem_bytes(e));
    A.rew_stride = (int64_t)(e->multi ? cells_all : (size_t)e->N);
    A.actions = actions_dev;
    A.obs = obs_dev;
    A.reward = reward_dev;
    if (info) {
        A.info = *info;
        A.has_info = (info->demand_dev || info->ship_dev || info->acquisition_dev || info->order_dev || info->profit_dev) ? 1 : 0;
    }
    // fast path: whole tiles of E envs through the TMA-staged kernel; the tail (and configurations the
    // bulk copies cannot address: unaligned caller buffers, N not a multiple of 4) through the direct kernel
    const auto aligned16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
    const bool tma_legal = e->tma_fn && e->step_path != 1 && (e->N % 4) == 0 && aligned16(actions_dev) && aligned16(obs_dev) &&
                           aligned16(reward_dev);
    bool use_jit = false;
    const imxjit::Kernels* jk = nullptr;
    bool with_cc = false;
    if (cc_fused) *cc_fused = false;
    if (cc && tma_legal && !A.has_info && obs_dev && aligned16(cc->dev) && tile_io_whole16(e, e->tile_cc, true)) {
        if (e->jit_cc_state == 0 && !stream_is_capturing(s)) ensure_jit_cc(e);
        const int64_t whole = (e->N / e->tile_cc.E) * e->tile_cc.E;
        if (e->jit_cc_state == 1 && whole == e->N) {       // fused only when every env sits in a whole tile (else: unfused fallback)
            jk = e->jit_cc;
            use_jit = with_cc = true;
            A.cc = cc->dev; A.cc_fill = cc->fill; A.cc_lo = cc->lo; A.cc_hi = cc->hi;
            A.cc_W = (e->m - 1) * (1 + e->O) + e->O;
            if (cc_fused) *cc_fused = true;
        }
    }
    if (!with_cc && tma_legal && !A.has_info) {
        // the specialised kernels were loaded by imx_create() / imx_prepare(); the obs-less variant may still be
        // compiled here on first use, but never while the stream is being captured (module loads are not capturable)
        if (obs_dev) { if (e->jit_state == 1) jk = e->jit; }
        else {
            if (e->jit_noobs_state == 0 && !stream_is_capturing(s)) ensure_jit_noobs(e);
            if (e->jit_noobs_state == 1) jk = e->jit_noobs;
            else if (e->jit_state == 1 && e->jit_noobs_state == 0) jk = nullptr;   // capture in progress: ahead-of-time kernel
        }
        use_jit = jk != nullptr;
    }
    const TileLayout& TL_use = with_cc ? e->tile_cc : use_jit ? e->tile_jit : e->tile;
    const int epw_direct = 32 / e->m_pad;
    int64_t n_tma = 0;
    if (tma_legal && (with_cc || tile_io_whole16(e, TL_use, false))) {
        n_tma = (e->N / TL_use.E) * TL_use.E;
        while (n_tma > 0 && (n_tma % epw_direct) != 0) n_tma -= TL_use.E;      // the tail kernel starts on a warp-tile boundary
    }
    e->last_variant = 0;
    const bool fused = periods > 1 && n_tma == e->N && TL_use.total2 <= 200 * 1024 && e->fuse_periods;
    if (fused) A.periods = periods;
    if (done) *done = A.periods;
    const unsigned tma_smem = (unsigned)(fused ? TL_use.total2 : TL_use.total);
    if (n_tma > 0) {
        if (use_jit) {
            // persistent pipelined kernel (imx_step_pipe.cuh): a resident CTA walks over its tiles through a ring of stages
            PipeArgs PA;
            PA.n_tiles = (int32_t)(n_tma / TL_use.E);
            PA.stages = pipe_stages_for(e, TL_use);
            const bool pipe = !fused && jk->step_pipe && e->pipe_mode >= 0 && (e->pipe_mode == 1 || pipe_pays(e, PA.n_tiles));
            void* params[] = {(void*)&A, (void*)&TL_use, (void*)&PA};
            CUlaunchConfig lc;
            memset(&lc, 0, sizeof(lc));
            lc.gridDimX = (unsigned)(n_tma / TL_use.E); lc.gridDimY = 1; lc.gridDimZ = 1;
            const unsigned jthreads = (unsigned)((with_cc && e->step_et) ? e->tma_threads : e->jit_threads);
            lc.blockDimX = jthreads; lc.blockDimY = 1; lc.blockDimZ = 1;
            lc.sharedMemBytes = tma_smem;
            if (pipe) {
                const int64_t resident = (int64_t)e->sm_count * pipe_ctas_for(e, TL_use);
                lc.gridDimX = (unsigned)(PA.n_tiles < resident ? PA.n_tiles : resident);
                lc.blockDimX = jthreads + 32;
                lc.sharedMemBytes = (unsigned)(PA.stages * TL_use.total);
            }
            lc.hStream = (CUstream)s;
            CUlaunchAttribute at[1];
            at[0].id = CU_LAUNCH_ATTRIBUTE_PROGRAMMATIC_STREAM_SERIALIZATION;
            at[0].value.programmaticStreamSerializationAllowed = 1;
            lc.attrs = at;
            lc.numAttrs = e->use_pdl ? 1 : 0;
            const CUresult cr = imxjit::g_api.LaunchKernelEx(&lc, pipe ? jk->step_pipe : fused ? jk->step_many : jk->step, params, nullptr);
            if (cr != CUDA_SUCCESS) return fail(-3, "launch of the specialised step kernel failed (CUresult %d)", (int)cr);
            g_launches.fetch_add(1, std::memory_order_relaxed);
            e->last_variant = pipe ? 3 : 2;
        } else {
            cudaLaunchConfig_t lc;
            memset(&lc, 0, sizeof(lc));
            lc.gridDim = dim3((unsigned)(n_tma / TL_use.E));
            lc.blockDim = dim3((unsigned)e->tma_threads);
            lc.dynamicSmemBytes = (size_t)tma_smem;
            lc.stream = s;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            at[0].val.programmaticStreamSerializationAllowed = 1;
            lc.attrs = at;
            lc.numAttrs = e->use_pdl ? 1 : 0;
            IMX_CUDA(cudaLaunchKernelEx(&lc, fused ? e->tma_many_fn : e->tma_fn, A, e->tile));
            IMX_CHECK_LAUNCH("step_kernel_tma");
            e->last_variant = 1;
        }
    }
    if (n_tma < e->N) {
        A.n_begin = n_tma;
        const int epw = 32 / e->m_pad;
        const int64_t warp_tiles = (e->N - n_tma + epw - 1) / epw;
        const int64_t blocks_needed = (warp_tiles + (STEP_THREADS / 32) - 1) / (STEP_THREADS / 32);
        const unsigned grid = (unsigned)(blocks_needed < e->step_grid_cap ? blocks_needed : e->step_grid_cap);
        e->step_fn<<<grid, STEP_THREADS, e->step_smem, s>>>(A);
        IMX_CHECK_LAUNCH("step_kernel");
    }
    e->t += A.periods;
    return 0;
}

extern "C" int imx_step(imx_env* e, const void* actions_dev, void* obs_dev, double* reward_dev,
                        const imx_info_out* info, void* stream) {
    IMX_NVTX("imx_step");

    if (!e || !actions_dev || !reward_dev) return fail(-1, "null argument");
    IMX_CUDA(cudaSetDevice(e->cfg.device));
    return launch_step(e, actions_dev, (double*)obs_dev, reward_dev, info, (cudaStream_t)stream);
}

// step() that also emits the centralised-critic observation rows.  Fused into the step kernel's epilogue wherever the
// runtime-specialised TMA kernels serve the whole batch; otherwise the plain step followed by the gather kernel.
extern "C" int imx_step_cc(imx_env* e, const void* actions_dev, void* obs_dev, void* cc_dev, int fill_actions, double clip_lo,
                           double clip_hi, double* reward_dev, void* stream) {
    IMX_NVTX("imx_step_cc");

    if (!e || !actions_dev || !reward_dev || !cc_dev) return fail(-1, "null argument");
    if (!e->multi) return fail(-1, "the centralised-critic observation is defined for the multi-agent kinds");
    IMX_CUDA(cudaSetDevice(e->cfg.device));
    cudaStream_t s = (cudaStream_t)stream;
    void* obs = obs_dev;
    if (!obs) {                                              // the rows are built from the observation tile either way
        if (!e->d_obs_scratch) {
            if (stream_is_capturing(s)) return fail(-1, "imx_step_cc without obs_dev under stream capture: call imx_prepare(IMX_PREPARE_CC) first");
            IMX_CUDA(cudaMalloc(&e->d_obs_scratch, (size_t)e->N * e->m * e->O * obs_elem_bytes(e)));
        }
        obs = e->d_obs_scratch;
    }
    const CcOut cc = {cc_dev, fill_actions ? 1 : 0, clip_lo, clip_hi};
    bool fused = false;
    const int rc = launch_step(e, actions_dev, (double*)obs, reward_dev, nullptr, s, 1, nullptr, &cc, &fused);
    if (rc || fused) return rc;
    return imx_cc_observe(e, obs, fill_actions ? actions_dev : nullptr, clip_lo, clip_hi, cc_dev, obs_type_of(e->cfg), stream);
}

static int ensure_host_path(imx_env* e);

extern "C" int imx_prepare(imx_env* e, int flags) {
    if (!e) return fail(-1, "null env");
    IMX_CUDA(cudaSetDevice(e->cfg.device));
    // (0 keeps meaning the five flags it always meant: IMX_PREPARE_EPISODE compiles two more modules and is asked for explicitly)
    if (flags == 0) flags = IMX_PREPARE_STEP | IMX_PREPARE_NOOBS | IMX_PREPARE_HOST | IMX_PREPARE_DFO | IMX_PREPARE_CC;
    if (flags & IMX_PREPARE_STEP) ensure_jit(e);
    if (flags & IMX_PREPARE_NOOBS) ensure_jit_noobs(e);
    if (flags & IMX_PREPARE_HOST) { const int rc = ensure_host_path(e); if (rc) return rc; }
    if ((flags & IMX_PREPARE_CC) && e->multi) {
        ensure_jit_cc(e);
        if (!e->d_obs_scratch) IMX_CUDA(cudaMalloc(&e->d_obs_scratch, (size_t)e->N * e->m * e->O * obs_elem_bytes(e)));
    }
    if ((flags & IMX_PREPARE_DFO) && !e->multi && !e->d_dfo_rewards)
        IMX_CUDA(cudaMalloc(&e->d_dfo_rewards, (size_t)e->T * e->N * sizeof(double)));
    if (flags & IMX_PREPARE_EPISODE) {                     // both episode modules + every scratch buffer of the unfused form
        ensure_jit_episode(e, true);
        ensure_jit_episode(e, false);
        const size_t cols = e->multi ? e->m : 1, cells = (size_t)e->N * e->m;
        if (!e->d_ep_rewards) IMX_CUDA(cudaMalloc(&e->d_ep_rewards, (size_t)e->T * e->N * cols * sizeof(double)));
        if (!e->d_ep_profit) IMX_CUDA(cudaMalloc(&e->d_ep_profit, cells * sizeof(double)));
        if (!e->d_ep_ret) IMX_CUDA(cudaMalloc(&e->d_ep_ret, (size_t)e->N * cols * sizeof(double)));
        if (!e->d_ep_stats) IMX_CUDA(cudaMalloc(&e->d_ep_stats, (3 + 2 * (size_t)e->m) * sizeof(double)));
        if (!e->d_obs_scratch) IMX_CUDA(cudaMalloc(&e->d_obs_scratch, cells * e->O * obs_elem_bytes(e)));
    }
    IMX_CUDA(cudaDeviceSynchronize());
    return 0;
}

// K consecutive periods on pre-computed actions: one launch that keeps every tile's state in shared memory for all K
// periods (actions / demand prefetched two periods ahead, observations / rewards streamed out behind the compute)
// wherever the whole batch goes through the TMA kernel; otherwise K plain launches.  Same results either way.
extern "C" int imx_step_many(imx_env* e, const void* actions_dev, int K, void* obs_dev, double* reward_dev,
                             const imx_info_out* info, void* stream) {
    IMX_NVTX("imx_step_many");

    if (!e || !actions_dev || !reward_dev) return fail(-1, "null argument");
    if (K < 1) return fail(-1, "K must be >= 1");
    if (e->t + K > e->T) return fail(-6, "imx_step_many: %d periods from period %d run past the end of the episode (%d)", K, e->t, e->T);
    IMX_CUDA(cudaSetDevice(e->cfg.device));
    const size_t cells = (size_t)e->N * e->m;
    const size_t obs_stride = cells * e->O * obs_elem_bytes(e), act_stride = cells * act_elem_bytes(e);
    const size_t rew_stride = e->multi ? cells : (size_t)e->N;
    int j = 0;
    while (j < K) {
        int adv = 1;
        imx_info_out at;                                   // the diagnostics blocks of period j
        if (info) {
            at.demand_dev = info->demand_dev ? info->demand_dev + (size_t)j * cells : nullptr;
            at.ship_dev = info->ship_dev ? info->ship_dev + (size_t)j * cells : nullptr;
            at.acquisition_dev = info->acquisition_dev ? info->acquisition_dev + (size_t)j * cells : nullptr;
            at.order_dev = info->order_dev ? info->order_dev + (size_t)j * cells : nullptr;
            at.profit_dev = info->profit_dev ? info->profit_dev + (size_t)j * cells : nullptr;
        }
        const int rc = launch_step(e, (const unsigned char*)actions_dev + (size_t)j * act_stride,
                                   obs_dev ? (double*)((unsigned char*)obs_dev + (size_t)j * obs_stride) : nullptr,
                                   reward_dev + (size_t)j * rew_stride, info ? &at : nullptr, (cudaStream_t)stream, K - j, &adv);
        if (rc) return rc;
        j += adv;
    }
    return 0;
}

static int launch_return_stats(imx_env* e, const double* src, int periods, bool fused, double* ret_out, double* stats_dev, int accumulate,
                               cudaStream_t s);

// A whole stored-plan episode: reset + T steps + returns / statistics / evaluation accumulators.  One launch of the episode
// kernel (plus the two statistics launches over the returns) wherever the runtime-specialised build serves the whole batch
// with one tile per CTA; otherwise the composition of the existing calls, with the same results.
extern "C" int imx_replay_episode(imx_env* e, const int32_t* demand_dev, const uint8_t* delay_mask_dev, int noisy, uint64_t episode,
                                  const double* actions_dev, void* obs_dev, double* reward_dev, double* return_dev,
                                  double* stats_dev, int accumulate, double* eval_acc_dev, void* stream) {
    IMX_NVTX("imx_replay_episode");

    if (!e || !actions_dev) return fail(-1, "null argument");
    if ((noisy || delay_mask_dev) && !e->has_carry) return fail(-1, "noisy delay requested but the env was created with noisy_delay = 0");
    if (!demand_dev && e->cfg.demand_dist == IMX_DIST_REPLAY_ONLY)
        return fail(-1, "imx_replay_episode without a demand trace needs demand_dist poisson or uniform");
    IMX_CUDA(cudaSetDevice(e->cfg.device));
    cudaStream_t s = (cudaStream_t)stream;
    const bool capturing = stream_is_capturing(s);
    const int64_t N = e->N;
    const int m = e->m;
    const size_t cols = e->multi ? m : 1, cells = (size_t)N * m, es = obs_elem_bytes(e), aes = act_elem_bytes(e);
    if (!capturing) ensure_jit_episode(e, obs_dev != nullptr);
    const imxjit::Kernels* jk = obs_dev ? e->jit_ep : e->jit_ep_noobs;
    EpisodeArgs EA;
    memset(&EA, 0, sizeof(EA));
    const int64_t smem = episode_layout(e, EA, return_dev || stats_dev, eval_acc_dev != nullptr);
    const int64_t E = e->tile_jit.E;
    const auto aligned16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
    // the legality of imx_step_many's fused form (whole tiles, N % 4, 16-byte aligned buffers, a layout that fits), and the
    // replayed trace's per-tile block [E][R][T] must be a whole number of 16-byte units
    // divergent networks (measured, profiles/r3_replay_episode.jsonl): the episode kernel is ahead where the period body is the
    // env-per-thread one and observations are written (div2 +3 %), and where it is lane-mapped without observations (div1 +1 to
    // +6 %); in the other two cases its larger resident layout costs more than the bookkeeping it saves (div2 without observations
    // -7 to -12 %, div1 with observations -6 % at 32 768 envs), so the composition serves them
    const bool pays = !e->div || (e->step_et ? obs_dev != nullptr : obs_dev == nullptr);
    const bool fused = pays && jk && jk->step_episode && e->step_path != 1 && e->fuse_periods && N % 4 == 0 && N % E == 0 && E % 2 == 0 &&
                       smem <= 200 * 1024 && tile_io_whole16(e, e->tile_jit, false) && aligned16(actions_dev) && aligned16(obs_dev) && aligned16(reward_dev) && aligned16(return_dev) &&
                       aligned16(eval_acc_dev) && (!demand_dev || (aligned16(demand_dev) && (E * e->R * e->T) % 4 == 0));
    // internal buffers are allocated here (never under capture: imx_prepare(IMX_PREPARE_EPISODE) allocates them up front),
    // before anything is launched
    auto scratch = [&](void** p, size_t bytes) -> int {
        if (*p) return 0;
        if (capturing) return fail(-1, "imx_replay_episode needs an internal buffer under stream capture: call imx_prepare(IMX_PREPARE_EPISODE) first");
        IMX_CUDA(cudaMalloc(p, bytes));
        return 0;
    };
    int rc = 0;
    if (fused) {
        double* ret = return_dev;
        if (!ret && stats_dev) {                              // the statistics read the returns: keep them in a scratch row
            if ((rc = scratch((void**)&e->d_ep_ret, (size_t)N * cols * sizeof(double)))) return rc;
            ret = e->d_ep_ret;
        }
        StepArgs A;
        fill_args(e, A);
        A.t = 0;
        A.noisy = (noisy || delay_mask_dev) ? 1 : 0;
        A.periods = e->T;
        A.act_stride = (int64_t)cells;
        A.obs_stride_bytes = (int64_t)(cells * e->O * es);
        A.rew_stride = (int64_t)(N * cols);
        A.actions = actions_dev;
        A.obs = (double*)obs_dev;
        A.reward = reward_dev;
        EA.demand = demand_dev;
        EA.mask = delay_mask_dev;
        EA.ret = ret;
        EA.eval = eval_acc_dev;
        EA.gen = make_gen(e, episode);
        EA.delay_thr = e->cfg.noisy_delay_threshold;
        EA.rescaled = (e->cfg.kind == IMX_KIND_MAIM_DIV || e->cfg.standardise_state) ? 1 : 0;
        void* params[] = {(void*)&A, (void*)&e->tile_jit, (void*)&EA};
        CUlaunchConfig lc;
        memset(&lc, 0, sizeof(lc));
        lc.gridDimX = (unsigned)(N / E); lc.gridDimY = 1; lc.gridDimZ = 1;
        lc.blockDimX = (unsigned)e->jit_threads; lc.blockDimY = 1; lc.blockDimZ = 1;
        lc.sharedMemBytes = (unsigned)smem;
        lc.hStream = (CUstream)s;
        CUlaunchAttribute at[1];
        at[0].id = CU_LAUNCH_ATTRIBUTE_PROGRAMMATIC_STREAM_SERIALIZATION;
        at[0].value.programmaticStreamSerializationAllowed = 1;
        lc.attrs = at;
        lc.numAttrs = e->use_pdl ? 1 : 0;
        const CUresult cr = imxjit::g_api.LaunchKernelEx(&lc, jk->step_episode, params, nullptr);
        if (cr != CUDA_SUCCESS) return fail(-3, "launch of the episode kernel failed (CUresult %d)", (int)cr);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        e->last_variant = 4;
        e->t = e->T;
        e->episode = episode;
        e->noisy_now = A.noisy;
        return stats_dev ? launch_return_stats(e, ret, 1, false, nullptr, stats_dev, accumulate, s) : 0;
    }
    // the composition: imx_reset + imx_step_many (per-period steps with the profit diagnostics when the accumulators are
    // wanted) + imx_episode_stats
    double* rew = reward_dev;
    if (!rew && (rc = scratch((void**)&e->d_ep_rewards, (size_t)e->T * N * cols * sizeof(double)))) return rc;
    if (!rew) rew = e->d_ep_rewards;
    if (eval_acc_dev) {
        if ((rc = scratch((void**)&e->d_ep_profit, cells * sizeof(double)))) return rc;
        if (!obs_dev && (rc = scratch(&e->d_obs_scratch, cells * e->O * es))) return rc;
    }
    double* st = stats_dev;
    if (!st && return_dev) {
        if ((rc = scratch((void**)&e->d_ep_stats, (3 + 2 * (size_t)m) * sizeof(double)))) return rc;
        st = e->d_ep_stats;
        accumulate = 0;
    }
    if ((rc = imx_reset(e, demand_dev, delay_mask_dev, noisy, episode, nullptr, stream))) return rc;
    const size_t rstride = (size_t)N * cols;
    if (!eval_acc_dev) {
        if ((rc = imx_step_many(e, actions_dev, e->T, obs_dev, rew, nullptr, stream))) return rc;
    } else {
        for (int t = 0; t < e->T; ++t) {
            imx_info_out info;
            memset(&info, 0, sizeof(info));
            info.profit_dev = e->d_ep_profit;
            void* ob = obs_dev ? (void*)((unsigned char*)obs_dev + (size_t)t * cells * e->O * es) : e->d_obs_scratch;
            if ((rc = launch_step(e, (const unsigned char*)actions_dev + (size_t)t * cells * aes, (double*)ob, rew + (size_t)t * rstride, &info, s))) return rc;
            if ((rc = imx_eval_accumulate(e, ob, rew + (size_t)t * rstride, e->d_ep_profit, eval_acc_dev, t == 0, stream))) return rc;
        }
    }
    if (st) return imx_episode_stats(e, rew, e->T, return_dev, st, accumulate, stream);
    return 0;
}

// --------------------------------------------------------------------------------------
// fused base-stock rollout
// --------------------------------------------------------------------------------------
extern "C" int imx_rollout_basestock(imx_env* e, const double* z_dev, int z_stride, const int32_t* demand_dev,
                                     const uint8_t* delay_mask_dev, int noisy, uint64_t episode, const double* pmf_dev,
                                     double* return_dev, double* step_reward_dev, double* dfo_dev, int write_state, void* stream) {
    IMX_NVTX("imx_rollout_basestock");

    if (!e || !z_dev || !return_dev) return fail(-1, "null argument");
    if (z_stride != 0 && z_stride != e->m) return fail(-1, "z_stride must be 0 or m");
    if (dfo_dev && (!pmf_dev || e->multi)) return fail(-1, "dfo output needs pmf_dev and a single-agent kind");
    if (!demand_dev && e->cfg.demand_dist == IMX_DIST_REPLAY_ONLY)
        return fail(-1, "rollout without a demand trace needs demand_dist poisson or uniform");
    if ((noisy || delay_mask_dev) && !e->has_carry) return fail(-1, "noisy delay requested but the env was created with noisy_delay = 0");
    cudaStream_t s = (cudaStream_t)stream;
    IMX_CUDA(cudaSetDevice(e->cfg.device));
    if (dfo_dev && !step_reward_dev) {                       // the objective is a second kernel over the per-period rewards
        if (!e->d_dfo_rewards) {
            if (stream_is_capturing(s)) return fail(-1, "dfo_dev without step_reward_dev under stream capture: call imx_prepare(IMX_PREPARE_DFO) first");
            IMX_CUDA(cudaMalloc(&e->d_dfo_rewards, (size_t)e->T * e->N * sizeof(double)));
        }
        step_reward_dev = e->d_dfo_rewards;
    }
    StepArgs A;
    fill_args(e, A);
    A.t = 0;
    RolloutArgs Rg;
    memset(&Rg, 0, sizeof(Rg));
    Rg.z = z_dev; Rg.z_stride = z_stride; Rg.demand = demand_dev;
    Rg.ret = return_dev; Rg.step_reward = step_reward_dev; Rg.write_state = write_state;
    Rg.mask = delay_mask_dev; Rg.noisy = (noisy || delay_mask_dev) ? 1 : 0; Rg.delay_thr = e->cfg.noisy_delay_threshold;
    Rg.gen = make_gen(e, episode);
    const int epw = 32 / e->m_pad;
    // Philox demand is drawn cooperatively by the tile's lanes into shared memory when the episode fits
    const size_t draw_bytes = (size_t)(ROLLOUT_THREADS / 32) * epw * e->R * ((e->T + 1) & ~1) * sizeof(int32_t);
    const bool coop = (!demand_dev && draw_bytes <= 40 * 1024);
    Rg.coop_demand = coop ? 1 : 0;
    const size_t roll_smem = coop ? draw_bytes : 0;
    const int64_t warp_tiles = (e->N + epw - 1) / epw;
    const int64_t blocks_needed = (warp_tiles + (ROLLOUT_THREADS / 32) - 1) / (ROLLOUT_THREADS / 32);
    const unsigned grid = (unsigned)(blocks_needed < e->rollout_grid_cap ? blocks_needed : e->rollout_grid_cap);
    if (e->jit_state == 1 && e->jit->rollout && e->rollout_et) {
        EtNodeConsts C;
        memset(&C, 0, sizeof(C));
        for (int i = 0; i < e->m; ++i) {
            C.p[i] = e->sell[i]; C.c[i] = e->buy[i]; C.h[i] = e->cfg.stock_cost[i]; C.bc[i] = e->cfg.backlog_cost[i]; C.target[i] = e->cfg.inv_target[i];
        }
        void* params[] = {(void*)&A, (void*)&Rg, (void*)&C};
        const int64_t blocks = (e->N + ET_THREADS_HOST - 1) / ET_THREADS_HOST;
        const int64_t cap = (int64_t)e->sm_count * 16;
        Rg.coop_demand = 0;
        const CUresult cr = imxjit::g_api.LaunchKernel(e->jit->rollout, (unsigned)(blocks < cap ? blocks : cap), 1, 1, ET_THREADS_HOST, 1, 1, 0, (CUstream)s,
                                                       params, nullptr);
        if (cr != CUDA_SUCCESS) return fail(-3, "launch of the env-per-thread rollout kernel failed (CUresult %d)", (int)cr);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        e->last_variant = 2;
    } else if (e->jit_state == 1 && e->jit->rollout) {
        void* params[] = {(void*)&A, (void*)&Rg};
        const int epw_j = 32 / e->m;                         // dense packing in the specialised build
        const int64_t wt_j = (e->N + epw_j - 1) / epw_j;
        const int64_t need_j = (wt_j + (ROLLOUT_THREADS / 32) - 1) / (ROLLOUT_THREADS / 32);
        const int64_t cap_j = (int64_t)e->rollout_grid_cap * 4;
        const unsigned g2 = (unsigned)(need_j < cap_j ? need_j : cap_j);
        const size_t draw_j = (size_t)(ROLLOUT_THREADS / 32) * epw_j * e->R * ((e->T + 1) & ~1) * sizeof(int32_t);
        if (coop && draw_j > 40 * 1024) Rg.coop_demand = 0;
        const size_t roll_smem_j = Rg.coop_demand ? draw_j : 0;
        const CUresult cr = imxjit::g_api.LaunchKernel(e->jit->rollout, g2, 1, 1, ROLLOUT_THREADS, 1, 1, (unsigned)roll_smem_j, (CUstream)s, params, nullptr);
        if (cr != CUDA_SUCCESS) return fail(-3, "launch of the specialised rollout kernel failed (CUresult %d)", (int)cr);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        e->last_variant = 2;
    } else {
        e->rollout_fn<<<grid, ROLLOUT_THREADS, roll_smem, s>>>(A, Rg);
        IMX_CHECK_LAUNCH("rollout_kernel");
        e->last_variant = 0;
    }
    if (dfo_dev) {
        dfo_objective_kernel<<<(unsigned)((e->N + 127) / 128), 128, 0, s>>>(pmf_dev, step_reward_dev, dfo_dev, e->N, e->R, e->T);
        IMX_CHECK_LAUNCH("dfo_objective_kernel");
    }
    if (write_state) { e->t = e->T; e->episode = episode; e->noisy_now = Rg.noisy; }
    return 0;
}

// launches `kern` as a programmatic dependent of the kernel in front of it on the stream (the kernel itself starts with
// griddepcontrol.wait): its launch latency overlaps the predecessor's tail
template <typename... KArgs, typename... Args>
static cudaError_t launch_dependent(void (*kern)(KArgs...), dim3 grid, dim3 block, cudaStream_t s, bool pdl, Args... args) {
    cudaLaunchConfig_t lc;
    memset(&lc, 0, sizeof(lc));
    lc.gridDim = grid; lc.blockDim = block; lc.dynamicSmemBytes = 0; lc.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = at;
    lc.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&lc, kern, KArgs(args)...);
}

// stage 1 (one block per slice of envs; FUSED adds the step rewards first) + stage 2 of the return statistics
static int launch_return_stats(imx_env* e, const double* src, int periods, bool fused, double* ret_out, double* stats_dev, int accumulate,
                               cudaStream_t s) {
    const int cols = e->multi ? e->m : 1;
    const int per_agent = e->multi ? 1 : 0;
    const int nstat = per_agent ? 2 + 2 * cols : 2;
    const int epb = stats_envs_per_block(cols);
    const int nslices = (int)((e->N + epb - 1) / epb);
    const bool pdl = e->use_pdl != 0;
    // one row of "step rewards" whose sum nobody asked for IS the returns: the plain kernel keeps four loads per thread in flight
    if (fused && periods == 1 && !ret_out) fused = false;
    if (fused)
        IMX_CUDA(launch_dependent(stats_slice_kernel<true>, dim3((unsigned)nslices), dim3(STATS_THREADS), s, pdl, src, ret_out, e->d_stats_partial,
                                  e->N, cols, per_agent, periods, epb, nslices));
    else
        IMX_CUDA(launch_dependent(stats_slice_kernel<false>, dim3((unsigned)nslices), dim3(STATS_THREADS), s, pdl, src, (double*)nullptr,
                                  e->d_stats_partial, e->N, cols, per_agent, 1, epb, nslices));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    IMX_CUDA(launch_dependent(stats_final_kernel, dim3((unsigned)nstat), dim3(STATS_THREADS), s, pdl, (const double*)e->d_stats_partial, stats_dev,
                              e->N, nslices, accumulate));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

extern "C" int imx_return_stats(imx_env* e, const double* return_dev, double* stats_dev, void* stream) {
    if (!e || !return_dev || !stats_dev) return fail(-1, "null argument");
    IMX_CUDA(cudaSetDevice(e->cfg.device));
    return launch_return_stats(e, return_dev, 1, false, nullptr, stats_dev, 0, (cudaStream_t)stream);
}

extern "C" int imx_episode_stats(imx_env* e, const double* step_reward_dev, int periods, double* return_dev, double* stats_dev,
                                 int accumulate, void* stream) {
    IMX_NVTX("imx_episode_stats");

    if (!e || !step_reward_dev || !stats_dev) return fail(-1, "null argument");
    if (periods < 1) return fail(-1, "periods must be >= 1");
    IMX_CUDA(cudaSetDevice(e->cfg.device));
    // the episode returns are only written when the caller asks for them (the statistics are built from shared memory)
    return launch_return_stats(e, step_reward_dev, periods, true, return_dev, stats_dev, accumulate, (cudaStream_t)stream);
}

// --------------------------------------------------------------------------------------
// evaluation-loop accumulators (MA_inv_management.py:538-600 and its siblings)
// --------------------------------------------------------------------------------------
extern "C" int imx_eval_len(const imx_env* e) { return e ? EVAL_FIXED + e->m : -1; }

extern "C" int imx_eval_accumulate(imx_env* e, const void* obs_dev, const double* reward_dev, const double* profit_dev,
                                   double* acc_dev, int reset, void* stream) {
    if (!e || !obs_dev || !reward_dev || !acc_dev) return fail(-1, "null argument");
    IMX_CUDA(cudaSetDevice(e->cfg.device));
    EvalArgs E;
    memset(&E, 0, sizeof(E));
    E.obs = obs_dev; E.reward = reward_dev; E.profit = profit_dev; E.acc = acc_dev; E.nodes = e->d_nodes;
    E.N = e->N; E.m = e->m; E.O = e->O; E.multi = e->multi ? 1 : 0; E.obs_type = obs_type_of(e->cfg);
    E.rescaled = (e->cfg.kind == IMX_KIND_MAIM_DIV || e->cfg.standardise_state) ? 1 : 0;
    E.reset = reset ? 1 : 0;
    E.a = e->cfg.a; E.bma = e->cfg.b - e->cfg.a;
    eval_accumulate_kernel<<<(unsigned)((e->N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(E);
    IMX_CHECK_LAUNCH("eval_accumulate_kernel");
    return 0;
}

extern "C" int imx_eval_stats(imx_env* e, const double* acc_dev, double* stats_dev, int accumulate, void* stream) {
    if (!e || !acc_dev || !stats_dev) return fail(-1, "null argument");
    IMX_CUDA(cudaSetDevice(e->cfg.device));
    const int W = EVAL_FIXED + e->m;
    column_stats_partial_kernel<<<dim3(STATS_BLOCKS, 2 * W), STATS_THREADS, 0, (cudaStream_t)stream>>>(acc_dev, e->d_stats_partial, e->N, W);
    IMX_CHECK_LAUNCH("column_stats_partial_kernel");
    stats_final_kernel<<<2 * W, STATS_THREADS, 0, (cudaStream_t)stream>>>(e->d_stats_partial, stats_dev, e->N, STATS_BLOCKS, accumulate);
    IMX_CHECK_LAUNCH("stats_final_kernel");
    return 0;
}

// --------------------------------------------------------------------------------------
// host-buffer convenience path (end-to-end: H2D + kernels + D2H + sync)
// --------------------------------------------------------------------------------------
static int ensure_host_path(imx_env* e) {
    if (e->hstream) return 0;
    const size_t cells = (size_t)e->N * e->m;
    // the stream handle marks the path as ready, so it is published last: a failed allocation leaves nothing half-built
    cudaError_t rc = cudaSuccess;
    auto take = [&](void** p, size_t bytes) { if (rc == cudaSuccess && !*p) rc = cudaMalloc(p, bytes); };
    take((void**)&e->d_act_h, cells * sizeof(double));
    take((void**)&e->d_obs_h, cells * e->O * obs_elem_bytes(e));
    take((void**)&e->d_rew_h, cells * sizeof(double));
    take((void**)&e->d_dem_h, (size_t)e->N * e->R * e->T * sizeof(int32_t));
    if (e->has_carry) take((void**)&e->d_mask_h, (size_t)e->N * e->T * e->m);
    cudaStream_t hs = nullptr;
    if (rc == cudaSuccess) rc = cudaStreamCreateWithFlags(&hs, cudaStreamNonBlocking);
    if (rc != cudaSuccess) {
        cudaFree(e->d_act_h); cudaFree(e->d_obs_h); cudaFree(e->d_rew_h); cudaFree(e->d_dem_h); cudaFree(e->d_mask_h);
        e->d_act_h = e->d_obs_h = e->d_rew_h = nullptr; e->d_dem_h = nullptr; e->d_mask_h = nullptr;
        return fail(-2, "host-path staging allocation failed: %s", cudaGetErrorString(rc));
    }
    e->hstream = hs;
    return 0;
}

extern "C" int imx_reset_host(imx_env* e, const int32_t* demand_host, const uint8_t* delay_mask_host, int noisy,
                              uint64_t episode, void* obs_host) {
    IMX_NVTX("imx_reset_host");

    if (!e) return fail(-1, "null env");
    IMX_CUDA(cudaSetDevice(e->cfg.device));
    int rc = ensure_host_path(e);
    if (rc) return rc;
    cudaStream_t s = e->hstream;
    if (demand_host)
        IMX_CUDA(cudaMemcpyAsync(e->d_dem_h, demand_host, (size_t)e->N * e->R * e->T * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    if (delay_mask_host) {
        if (!e->has_carry) return fail(-1, "noisy delay requested but the env was created with noisy_delay = 0");
        IMX_CUDA(cudaMemcpyAsync(e->d_mask_h, delay_mask_host, (size_t)e->N * e->T * e->m, cudaMemcpyHostToDevice, s));
    }
    rc = imx_reset(e, demand_host ? e->d_dem_h : nullptr, delay_mask_host ? e->d_mask_h : nullptr, noisy, episode,
                   obs_host ? e->d_obs_h : nullptr, s);
    if (rc) return rc;
    if (obs_host)
        IMX_CUDA(cudaMemcpyAsync(obs_host, e->d_obs_h, (size_t)e->N * e->m * e->O * obs_elem_bytes(e), cudaMemcpyDeviceToHost, s));
    IMX_CUDA(cudaStreamSynchronize(s));
    return 0;
}

// Device-visible alias of a pinned (page-locked, mapped) host pointer under UVA, or NULL.
static void* pinned_alias(const void* host_ptr) {
    if (!host_ptr) return nullptr;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, host_ptr) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) return nullptr;
    return at.devicePointer;
}

extern "C" int imx_step_host(imx_env* e, const void* actions_host, void* obs_host, double* reward_host) {
    IMX_NVTX("imx_step_host");

    if (!e || !actions_host || !reward_host) return fail(-1, "null argument");
    IMX_CUDA(cudaSetDevice(e->cfg.device));
    int rc = ensure_host_path(e);
    if (rc) return rc;
    cudaStream_t s = e->hstream;
    const size_t cells = (size_t)e->N * e->m;
    // Zero-copy fast path: with pinned buffers the kernel's bulk loads / stores address host memory
    // directly over PCIe (UVA), so transfer and compute overlap tile by tile and no staging copy exists.
    const void* act_d = pinned_alias(actions_host);
    double* obs_d = obs_host ? (double*)pinned_alias(obs_host) : nullptr;
    double* rew_d = (double*)pinned_alias(reward_host);
    const bool zero_copy = e->host_zero_copy && act_d && rew_d && (obs_d || !obs_host);
    if (zero_copy) {
        // Over PCIe the direct kernel (persistent warps, one bulk store per warp tile) measured 3.6 % faster than the
        // TMA-tiled one (712 vs 687 M agent-steps/s at 65536 envs): the link, not the SM, is the bottleneck here.
        const int saved_path = e->step_path;
        if (saved_path == 0) e->step_path = 1;
        rc = launch_step(e, act_d, obs_d, rew_d, nullptr, s);
        e->step_path = saved_path;
        if (rc) return rc;
        IMX_CUDA(cudaStreamSynchronize(s));
        return 0;
    }
    IMX_CUDA(cudaMemcpyAsync(e->d_act_h, actions_host, cells * act_elem_bytes(e), cudaMemcpyHostToDevice, s));
    rc = launch_step(e, e->d_act_h, obs_host ? e->d_obs_h : nullptr, e->d_rew_h, nullptr, s);
    if (rc) return rc;
    if (obs_host) IMX_CUDA(cudaMemcpyAsync(obs_host, e->d_obs_h, cells * e->O * obs_elem_bytes(e), cudaMemcpyDeviceToHost, s));
    IMX_CUDA(cudaMemcpyAsync(reward_host, e->d_rew_h, (e->multi ? cells : (size_t)e->N) * sizeof(double), cudaMemcpyDeviceToHost, s));
    IMX_CUDA(cudaStreamSynchronize(s));
    return 0;
}

extern "C" int imx_poisson_cdf(const imx_env* e, double* out, int cap) {
    if (!e) return fail(-1, "null env");
    if (e->cfg.demand_dist != IMX_DIST_POISSON) return 0;
    if (out) {
        std::vector<double> cdf = poisson_cdf(e->cfg.mu);
        for (int k = 0; k < (int)cdf.size() && k < cap; ++k) out[k] = cdf[k];
    }
    return e->cdf_len;
}

// --------------------------------------------------------------------------------------
// kernel-variant introspection and the CPU-side check of the runtime-specialised build
// --------------------------------------------------------------------------------------
extern "C" int imx_kernel_variant(const imx_env* e) { return e ? e->last_variant : fail(-1, "null env"); }
extern "C" const char* imx_jit_log(void) { return imxjit::g_last_log.c_str(); }

extern "C" int imx_jit_compile_check(const imx_config* cfg, int variant, char* log, int cap) {
    if (!cfg) return fail(-1, "null argument");
    if (variant < 0 || variant > 4)
        return fail(-1, "variant must be 0 (step), 1 (no observations), 2 (critic rows), 3 (episode) or 4 (episode without observations)");
    imx_env tmp;
    tmp.cfg = *cfg;
    const int rc = derive(&tmp);
    if (rc) return rc;
    tmp.tma_threads = choose_tma_threads(&tmp);
    {
        const char* re = getenv("IMX_ROLLOUT_ET");
        tmp.rollout_et = (re && !strcmp(re, "0")) ? 0 : (tmp.m <= 8 && tmp.D <= 4);
        const char* se = getenv("IMX_STEP_ET");
        const bool et_ok = tmp.m <= 8 && tmp.D <= 4 && tmp.P <= 2;
        const bool non_pow2 = (tmp.m & (tmp.m - 1)) != 0;
        tmp.step_et = (se && !strcmp(se, "0")) ? 0 : (se && !strcmp(se, "1")) ? et_ok : (et_ok && tmp.div && non_pow2);
        const char* st = getenv("IMX_STEP_ET_THREADS");
        const int et_threads = (st && (atoi(st) == 32 || atoi(st) == 64 || atoi(st) == 128)) ? atoi(st) : 32;
        tmp.jit_threads = tmp.step_et ? et_threads : tmp.tma_threads;
        tmp.l2_hints = decide_l2_hints(&tmp, 0);
    }
    compute_tile(&tmp, tmp.tile, m_pad_of(&tmp));
    compute_tile(&tmp, tmp.tile_jit, m_pad_of(&tmp), false, tmp.step_et ? tmp.jit_threads : 0);
    compute_tile(&tmp, tmp.tile_cc, m_pad_of(&tmp), true);
    int TL = 0;
    build_tables(&tmp, &TL);
    imxjit::Spec sp;
    if (variant == 2 && !tmp.multi) return fail(-1, "the critic rows exist for the multi-agent kinds only");
    EpisodeArgs EA;
    if (variant >= 3 && episode_layout(&tmp, EA) > 200 * 1024) return fail(-1, "the episode kernel's layout exceeds 200 KB of shared memory");
    jit_spec(&tmp, TL, sp, (variant == 1 || variant == 4) ? 0 : 1, variant == 2 ? 1 : 0, variant >= 3 ? 1 : 0);
    std::string lg;
    std::vector<char> cubin;
    const size_t n = imxjit::compile_only(sp, lg, &cubin);
    if (n > 0 && getenv("IMX_JIT_DUMP")) {              // for cuobjdump -sass inspection
        FILE* f = fopen(getenv("IMX_JIT_DUMP"), "wb");
        if (f) { fwrite(cubin.data(), 1, cubin.size(), f); fclose(f); }
    }
    if (log && cap > 0) { strncpy(log, lg.c_str(), (size_t)cap - 1); log[cap - 1] = 0; }
    if (n == 0) return fail(-7, "runtime specialisation did not compile: %s", lg.substr(0, 300).c_str());
    return (int)n;
}

// --------------------------------------------------------------------------------------
// centralised-critic observation (models/CC_Model.py:165-214)
// --------------------------------------------------------------------------------------
extern "C" int imx_cc_obs_len(const imx_env* e) { return e ? (e->m - 1) * (1 + e->O) + e->O : fail(-1, "null env"); }

extern "C" int imx_cc_observe(imx_env* e, const void* obs_dev, const void* actions_dev, double clip_lo, double clip_hi,
                              void* out_dev, int out_is_f32, void* stream) {
    if (!e || !obs_dev || !out_dev) return fail(-1, "null argument");
    if (!e->multi) return fail(-1, "the centralised-critic observation is defined for the multi-agent kinds");
    if (out_is_f32 < 0 || out_is_f32 > 2) return fail(-1, "out_is_f32 must be 0 (float64), 1 (float32) or 2 (bfloat16)");
    IMX_CUDA(cudaSetDevice(e->cfg.device));
    const int W = (e->m - 1) * (1 + e->O) + e->O;
    const int64_t total = e->N * e->m * W;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->cfg.device);
    const int64_t want = (total + 255) / 256;
    const unsigned grid = (unsigned)(want < (int64_t)sms * 16 ? want : (int64_t)sms * 16);
    cudaStream_t s = (cudaStream_t)stream;
    const int af = act_elem_bytes(e) == 4 ? 1 : 0;
    // the observations are read in the element type the env writes, the rows written in the one asked for
    auto launch = [&](auto in_tag) {
        using InT = decltype(in_tag);
        const InT* in = (const InT*)obs_dev;
        if (out_is_f32 == 2) cc_observer_kernel<InT, Bf16><<<grid, 256, 0, s>>>(in, actions_dev, af, (Bf16*)out_dev, e->N, e->m, e->O, clip_lo, clip_hi);
        else if (out_is_f32) cc_observer_kernel<InT, float><<<grid, 256, 0, s>>>(in, actions_dev, af, (float*)out_dev, e->N, e->m, e->O, clip_lo, clip_hi);
        else cc_observer_kernel<InT, double><<<grid, 256, 0, s>>>(in, actions_dev, af, (double*)out_dev, e->N, e->m, e->O, clip_lo, clip_hi);
    };
    const int ot = obs_type_of(e->cfg);
    if (ot == OBS_BF16) launch(Bf16{});
    else if (ot == OBS_F32) launch(0.0f);
    else launch(0.0);
    IMX_CHECK_LAUNCH("cc_observer_kernel");
    return 0;
}
