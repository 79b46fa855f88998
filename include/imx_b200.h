/*
 * imx_b200.h — C ABI of the B200-native batched inventory-management environment step.
 *
 * Drop-in boundary for ONE hot path of MarwanMousa/MARL-for-IM: reset()/step() of
 *   environments/IM_env.py        InvManagement             (kind IMX_KIND_IM)
 *   environments/MAIM_env.py      MultiAgentInvManagement   (kind IMX_KIND_MAIM)
 *   environments/IM_div_env.py    InvManagementDiv          (kind IMX_KIND_IM_DIV)
 *   environments/MAIM_div_env.py  MultiAgentInvManagementDiv(kind IMX_KIND_MAIM_DIV)
 * and the rollout loop of base_restock_policy.py.  The reference has no FFI layer (it is
 * pure Python); each entry point below names the reference method it replaces.  A batch of
 * N independent environments advances in lock-step (episodes are fixed length, so the
 * period counter is a scalar of the batch, cf. MAIM_env.py:395-397).
 *
 * Conventions
 *   - plain C, no C++/torch types; every `_dev` pointer is caller-owned device memory on the
 *     env's device (e.g. a torch tensor's data_ptr()), valid until the stream work finishes;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - no entry point synchronises the device, allocates memory or loads code after imx_create() /
 *     imx_prepare(), except the *_host convenience calls and the first dfo_dev use of
 *     imx_rollout_basestock without a step_reward_dev buffer, so reset/step sequences can be captured
 *     in CUDA graphs.  The runtime-specialised kernels (NVRTC) are compiled and loaded inside
 *     imx_create() when the batch size selects them; a call issued under stream capture never compiles;
 *   - return value 0 = success, negative = error (imx_last_error() gives the message, thread
 *     local); nothing throws across the ABI;
 *   - one handle is not thread-safe; different handles are independent.
 *
 * Data layout (row-major, env index slowest unless stated)
 *   actions  [N][m] float64      reward (MAIM kinds) [N][m] float64, (IM kinds) [N] float64
 *   obs      [N][m][O] float64   row i of env n = agent i's observation vector (float32 when cfg.obs_f32)
 *   demand   [N][R][T] int32     replayed customer demand, R = number of retailers (serial: 1)
 *   mask     [N][T][m] uint8     replayed noisy-delay Bernoulli outcomes (u <= threshold)
 *   state    int32 structure-of-arrays, see imx_state_field()
 */
#ifndef IMX_B200_H
#define IMX_B200_H

#ifndef __CUDACC_RTC__
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define IMX_ABI_VERSION 3     /* 3: obs pointers are void* (float64, or float32 with cfg.obs_f32) everywhere; imx_rollout_basestock gained
                                 delay_mask_dev / noisy and takes pmf [N][R][T]; imx_prepare; imx_step_cc.
                                 2: imx_config gained obs_f32 + noisy_demand_threshold; imx_step_many, imx_eval_*; imx_cc_observe takes void* */
#define IMX_MAX_NODES 32     /* agents (stages / nodes) per env: one lane each            */
#define IMX_MAX_CHILDREN 8   /* children per node in a divergent network                  */
#define IMX_MAX_DELAY 8      /* lead time per stage (shipped configs use <= 4)            */
#define IMX_MAX_HIST 8       /* prev_length (shipped configs use 1..3)                    */

enum imx_kind { IMX_KIND_IM = 0, IMX_KIND_MAIM = 1, IMX_KIND_IM_DIV = 2, IMX_KIND_MAIM_DIV = 3 };
enum imx_demand_dist { IMX_DIST_REPLAY_ONLY = 0, IMX_DIST_POISSON = 1, IMX_DIST_UNIFORM = 2 };

/* Per-config constants.  The host mirrors the reference constructors
 * (IM_env.py:7-162, MAIM_env.py:8-173, IM_div_env.py:9-199, MAIM_div_env.py:9-237): it applies
 * the per-class defaults and passes explicit vectors; the library derives demand_max, the
 * depth-based node prices of the divergent envs, the observation length and the state layout. */
typedef struct imx_config {
    int32_t kind;                 /* enum imx_kind                                           */
    int32_t num_nodes;            /* m: num_stages (serial) / num_nodes (divergent)          */
    int32_t num_periods;          /* T                                                       */
    int32_t prev_length;          /* P                                                       */
    int32_t time_dependency;      /* obs carries the lead-time pipeline                      */
    int32_t prev_demand;          /* obs carries the last P demands                          */
    int32_t prev_actions;         /* obs carries the last P clipped orders                   */
    int32_t standardise_state;    /* ignored (treated as 1) for IMX_KIND_MAIM_DIV            */
    int32_t standardise_actions;  /* ignored (treated as 1) for IMX_KIND_MAIM_DIV            */
    int32_t independent;          /* MAIM kinds: per-agent profit (1) or shared mean (0)     */
    int32_t share_network;        /* MAIM_DIV: append the node-id feature                    */
    int32_t noisy_delay;          /* allocate the carry state; 0 = lead times are exact      */
    int32_t demand_dist;          /* enum imx_demand_dist: generator used when reset() gets no trace */
    int32_t uniform_low;          /* IMX_DIST_UNIFORM: integers in [low, high)               */
    int32_t uniform_high;
    int32_t device;               /* CUDA device ordinal                                      */
    int32_t obs_f32;              /* 1: observations are written as float32 (= the float32 cast of the reference's float64 value; RLlib casts anyway), obs buffers are [N][m][O] float */
    int32_t reserved0;
    double a, b;                  /* rescale interval (IM_DIV: the host passes -1, 1)        */
    double mu;                    /* IMX_DIST_POISSON mean                                   */
    double noisy_delay_threshold; /* used when the mask is generated (Philox) instead of replayed */
    double noisy_demand_threshold; /* divergent kinds, generated demand only (MAIM_div_env.py:287-295): each period's draw is
                                      doubled with this probability, then zeroed with this probability; 0 = off */
    uint64_t seed;                /* Philox key                                               */
    int64_t num_envs;             /* N: envs in this handle (this rank's shard)              */
    int64_t env_offset;           /* global index of local env 0 (Philox counter; makes results independent of sharding) */
    /* Capacities above 2^28 are refused, and so is any config whose int32 state could wrap (DESIGN.md §6): with dmax_i the
     * most node i can be asked for in one period (a retailer's inv_max, the downstream stage's order_max, the sum of the
     * children's order_max), demand_max must fit int32, and T * dmax_i must too wherever the backlog is uncapped
     * (standardise_state = 0 on IM / IM_DIV / MAIM) and for every divergent node with more than one child (its ledger).
     * With noisy_delay, inv_max_i + T * order_max_i (twice that for a divergent node other than 0) must fit int32 (the carry). */
    int32_t inv_init[IMX_MAX_NODES];
    int32_t inv_max[IMX_MAX_NODES];
    int32_t order_max[IMX_MAX_NODES];
    int32_t delay[IMX_MAX_NODES];                       /* >= 1, <= IMX_MAX_DELAY            */
    double inv_target[IMX_MAX_NODES];
    double stock_cost[IMX_MAX_NODES];
    double backlog_cost[IMX_MAX_NODES];
    double price[IMX_MAX_NODES + 1];                    /* serial kinds: price[i] sell, price[i+1] buy */
    int32_t num_children[IMX_MAX_NODES];                /* divergent kinds                    */
    int32_t children[IMX_MAX_NODES][IMX_MAX_CHILDREN];  /* in the order listed in `connections` (the split is order dependent) */
} imx_config;

typedef struct imx_env imx_env;   /* opaque */

/* Optional per-step diagnostics, replacing the `info` dict of step()
 * (MAIM_env.py:399-409, IM_env.py:345-350).  Any pointer may be NULL. */
typedef struct imx_info_out {
    int32_t* demand_dev;       /* [N][m] */
    int32_t* ship_dev;         /* [N][m] */
    int32_t* acquisition_dev;  /* [N][m] */
    int32_t* order_dev;        /* [N][m]  'actual order' */
    double*  profit_dev;       /* [N][m] */
} imx_info_out;

/* State fields for imx_state_field(): the persistent per-env state is exactly these int32
 * arrays (SURVEY.md appendix A.2); everything else in the reference's [T+1, m] arrays is history. */
enum imx_field {
    IMX_F_INV = 0,        /* [N][m]                                                          */
    IMX_F_BACKLOG = 1,    /* [N][m]                                                          */
    IMX_F_ORDER_U = 2,    /* [N][m]                                                          */
    IMX_F_PIPE = 3,       /* [N][L], L = sum(delay); stage i owns delay[i] consecutive slots, slot k arrives in k+1 periods */
    IMX_F_HIST_D = 4,     /* [N][m][P] last P demands (present iff the obs mode reads them)  */
    IMX_F_HIST_O = 5,     /* [N][m][P] last P clipped orders (iff prev_actions)              */
    IMX_F_CARRY = 6,      /* [N][m] goods held back one period by a noisy delay (iff noisy_delay) */
    IMX_F_BACKLOG_TO = 7, /* [N][NB] signed per-child backlog ledger of the split nodes, NB = sum of their child counts */
    IMX_F_ERROR = 8,      /* [N] watchdog code of the divergent split (0 = ok, 1..4 = "Infinite Loop k") */
    IMX_F_DEMAND = 9,     /* [T][R][N] the episode's demand trace as the kernels read it (transposed) */
    IMX_F_DELAY_MASK = 10, /* [T][N][m] uint8: this episode's noisy-delay outcomes (replayed or drawn from Philox) */
    IMX_F_COUNT = 11
};

#ifndef __CUDACC_RTC__   /* the device-side (NVRTC) build only needs the types above */
const char* imx_last_error(void);
int imx_abi_version(void);
int imx_config_size(void);   /* sizeof(imx_config): lets a foreign-language binding verify its struct mirror */

/* Env(config)  —  the constructors cited above.  Allocates all device state (zero further
 * allocations afterwards) and leaves the batch in the reset state with an all-zero demand trace. */
int imx_create(const imx_config* cfg, imx_env** out);
int imx_destroy(imx_env* env);

/* Loads every kernel variant this handle can dispatch to BEFORE the first step, so that no later call compiles,
 * loads a module or allocates (a requirement for capturing the first step() in a CUDA graph).  imx_create() already
 * does this for the variants its batch size selects; call imx_prepare() to force the rest.
 *   flags: IMX_PREPARE_STEP (observation-writing step / step_many / rollout kernels), IMX_PREPARE_NOOBS (the
 *          obs_dev = NULL specialisation), IMX_PREPARE_HOST (staging buffers + stream of the *_host calls),
 *          IMX_PREPARE_DFO (scratch of the dfo objective), IMX_PREPARE_CC (imx_step_cc's specialisation and scratch),
 *          IMX_PREPARE_EPISODE (imx_replay_episode's two episode kernels, with and without observations, and the scratch
 *          buffers of its unfused form: [T][N](m) rewards, [N][m][O] observations, [N][m] profits, [N](m) returns);
 *          0 = the first five (STEP | NOOBS | HOST | DFO | CC; not EPISODE, so existing callers compile nothing more).
 *          Synchronous; may take seconds (NVRTC). */
enum imx_prepare_flags { IMX_PREPARE_STEP = 1, IMX_PREPARE_NOOBS = 2, IMX_PREPARE_HOST = 4, IMX_PREPARE_DFO = 8, IMX_PREPARE_CC = 16,
                         IMX_PREPARE_EPISODE = 32 };
int imx_prepare(imx_env* env, int flags);

/* Derived sizes: O (observation length per agent), S (int32 state words per env), R, L, NB. */
int imx_obs_len(const imx_env* env);
int imx_state_words(const imx_env* env);
int imx_num_retailers(const imx_env* env);
int imx_pipe_words(const imx_env* env);
int imx_ledger_words(const imx_env* env);
int imx_retailers(const imx_env* env, int32_t* out /* [R] */);
int imx_demand_max(const imx_env* env, int32_t* out /* [m] */);
int imx_node_price(const imx_env* env, double* sell /* [m] */, double* buy /* [m] */);

/* Device pointer + element count of one state field (count 0 = field absent in this config). */
int imx_state_field(imx_env* env, int field, void** dev_ptr, int64_t* count);

/* Batch period counter (env.period).  Set it only to re-synchronise after replaying a captured graph. */
int imx_period(const imx_env* env);
int imx_set_period(imx_env* env, int t);

/* reset(customer_demand=None, noisy_delay=False, ...)  —  IM_env.py:164-229, MAIM_env.py:176-240,
 * IM_div_env.py:201-302, MAIM_div_env.py:240-341.
 *   demand_dev      replayed trace [N][R][T] int32, or NULL: draw Poisson/uniform demand from the
 *                   counter-based Philox stream keyed by (seed; global env, retailer, period, episode)
 *   delay_mask_dev  [N][T][m] uint8 replayed noisy-delay outcomes, or NULL: drawn from Philox with
 *                   noisy_delay_threshold when `noisy` is non-zero.  Needs cfg.noisy_delay = 1.
 *   noisy           0: exact lead times for this episode
 *   obs_dev         [N][m][O] receives the initial observation (may be NULL)                      */
int imx_reset(imx_env* env, const int32_t* demand_dev, const uint8_t* delay_mask_dev, int noisy,
              uint64_t episode, void* obs_dev, void* stream);

/* step(action)  —  IM_env.py:287-360, MAIM_env.py:330-411, IM_div_env.py:361-549,
 * MAIM_div_env.py:441-630: order clipping, demand propagation, acquisition, shipment (+ split),
 * backlog / pipeline / inventory update, profit reward, observation build.  One kernel launch.
 * done = imx_period(env) >= T after the call.  info may be NULL. */
int imx_step(imx_env* env, const double* actions_dev, void* obs_dev, double* reward_dev,
             const imx_info_out* info, void* stream);

/* K consecutive step() calls on pre-computed actions  —  the replay loops that drive an env with a stored plan
 * (the LP scripts: "lp_action = np.round(LP_actions[t, :], 0); s, r, done, info = LP_env.step(lp_action)",
 * DSHLP_4.py:905-908; evaluation of open-loop action traces).  Same results as K imx_step calls, bit for bit.
 * Where the whole batch goes through the TMA-staged kernel this is ONE launch: every tile's state stays in shared
 * memory for the K periods, actions / demand are prefetched two periods ahead and observations / rewards stream out
 * behind the compute, so state moves once per launch instead of once per period; otherwise K plain launches.
 *   actions_dev [K][N][m], obs_dev [K][N][m][O] or NULL, reward_dev [K][N][m] (MAIM kinds) / [K][N];
 *   info: NULL, or diagnostics arrays of K consecutive [N][m] blocks each (the array_profit / array_demand / array_ship /
 *   array_acquisition records of the LP replay loops, DSHLP_4.py:918-923). */
int imx_step_many(imx_env* env, const double* actions_dev, int K, void* obs_dev, double* reward_dev,
                  const imx_info_out* info, void* stream);

/* One whole episode on a stored plan: reset(customer_demand) + T step() calls + the episode's returns / statistics
 * (+ the evaluation loops' accumulators), i.e. the LP scripts' replay loop (DSHLP_4.py:896-928).  Bit-identical to
 *   imx_reset(env, demand_dev, delay_mask_dev, noisy, episode, NULL, s);
 *   imx_step_many(env, actions_dev, T, obs_dev, reward, NULL, s);                 (reward: reward_dev or scratch)
 *   imx_episode_stats(env, reward, T, return_dev, stats_dev, accumulate, s);       (when return_dev or stats_dev)
 *   imx_eval_accumulate(env, obs[t], reward[t], profit[t], eval_acc_dev, t == 0, s) for t < T   (when eval_acc_dev)
 * actions_dev [T][N][m]; obs_dev [T][N][m][O] or NULL; reward_dev [T][N][m] / [T][N] or NULL; return_dev [N][m] / [N] or NULL;
 * stats_dev [3 + 2m] / [3] or NULL; eval_acc_dev [N][4 + m] or NULL.  Leaves the env at period T with the final state
 * (every state field, the split's error flags).  demand_dev / delay_mask_dev / noisy / episode as in imx_reset: NULL draws
 * from the same Philox streams.  Works from any current period (it is a reset).
 * Where the runtime-specialised kernels serve the whole batch with one tile per CTA (N a multiple of the tile, 16-byte aligned
 * buffers, the tile's [E][R][T] trace fitting in shared memory) this is ONE kernel launch, plus the two statistics launches of
 * imx_return_stats when stats_dev is given; imx_kernel_variant() then returns 4.  That kernel reads the trace and the mask in
 * place, so on that path IMX_F_DEMAND and IMX_F_DELAY_MASK are NOT rewritten.  Elsewhere the library runs the composition
 * itself; its scratch buffers are allocated on first use, or by imx_prepare(IMX_PREPARE_EPISODE) — needed under capture. */
int imx_replay_episode(imx_env* env, const int32_t* demand_dev, const uint8_t* delay_mask_dev, int noisy, uint64_t episode,
                       const double* actions_dev, void* obs_dev, double* reward_dev, double* return_dev,
                       double* stats_dev, int accumulate, double* eval_acc_dev, void* stream);

/* dfo_func's loop  —  base_restock_policy.py:24-45 with base_stock_policy :4-21 fused in: a whole
 * K = T period episode per env in ONE kernel, state on chip.
 *   z_dev          base-stock levels, [m] (z_stride = 0) or [N][m] (z_stride = m)
 *   demand_dev     [N][R][T] replayed trace or NULL (Philox, same stream as imx_reset)
 *   delay_mask_dev [N][T][m] uint8 replayed noisy-delay outcomes or NULL; noisy != 0 with a NULL mask draws them
 *                  from Philox exactly as imx_reset(noisy = 1) of the same episode would.  The reference's noisy flag
 *                  is sticky (MAIM_env.py:192-194), so dfo_func after a noisy reset() rolls out WITH delays
 *                  (MAIM_env.py:449-457); needs cfg.noisy_delay = 1
 *   pmf_dev        optional [N][R][T] float64 probabilities of the demand trace (serial kinds: R = 1), or NULL
 *   return_dev     IM kinds [N], MAIM kinds [N][m]: sum over periods of the step reward
 *   step_reward_dev optional [T][N] (IM kinds) / [T][N][m] (MAIM kinds) per-period rewards, or NULL
 *   dfo_dev        optional [N]: -1 / T * np.sum(pmf * rewards) with the rewards broadcast over the R retailer rows and
 *                  numpy's pairwise summation order over the flattened [R, T] product, any R * T (needs pmf_dev; IM
 *                  kinds only — the reference's dfo_func cannot run on a dict-reward env).  A second small kernel over
 *                  step_reward_dev; when that is NULL an internal [T][N] scratch is allocated on first use
 *   write_state    non-zero: leave the final state in the env (period = T), else env is untouched */
int imx_rollout_basestock(imx_env* env, const double* z_dev, int z_stride, const int32_t* demand_dev,
                          const uint8_t* delay_mask_dev, int noisy, uint64_t episode, const double* pmf_dev,
                          double* return_dev, double* step_reward_dev, double* dfo_dev, int write_state, void* stream);

/* Episode statistics for the cross-GPU all-reduce: stats_dev[0..2] = {n, sum, sum of squares} of the
 * per-env total return, then per agent {sum, sum of squares} (MAIM kinds).  Deterministic order. */
int imx_return_stats(imx_env* env, const double* return_dev, double* stats_dev /* [3 + 2m] */, void* stream);

/* Statistics of one episode from its per-period rewards (the evaluation loops' "reward += r" then
 * np.mean / np.std over episodes): return[n][agent] = sum over periods in period order, then the
 * reduction of imx_return_stats.  step_reward_dev [periods][N][m] (MAIM kinds) / [periods][N];
 * return_dev [N][m] / [N] optional (only written when given); accumulate != 0 adds into stats_dev (an
 * evaluation batch builds up on the device, reduced across GPUs once).  Two launches (programmatic
 * dependents of whatever precedes them on the stream), no host work: graph-capturable. */
int imx_episode_stats(imx_env* env, const double* step_reward_dev, int periods, double* return_dev, double* stats_dev,
                      int accumulate, void* stream);

/* The evaluation loops' per-episode accumulators  —  MA_inv_management.py:538-587 (same loop:
 * CC_inv_management.py:512-556, CC_inv_management_div.py:500-544, inv_management.py:573-606, and the LP replay
 * loops, e.g. DSHLP_4.py:896-928).  Call once after every step() with that step's outputs:
 *   acc_dev [N][4 + m] float64 rows {episode_reward, total_inventory, total_backlog, customer_backlog,
 *           stage_profit[0..m-1]}: inventory/backlog are obs[.][0] / obs[.][1] mapped back with
 *           rev_scale(., 0, inv_max[stage], a, b) when the env standardises its state, summed over stages in
 *           stage order and then over periods, in float64, operation for operation like the host loop;
 *   profit_dev [N][m] (imx_info_out.profit_dev of the same step) or NULL: stage_profit columns stay as they are;
 *   reset != 0 starts a new episode (accumulators begin at zero).
 * imx_eval_stats reduces the rows to {n, then per column (sum, sum of squares)} = 1 + 2(4 + m) doubles, the
 * np.mean / np.std inputs of MA_inv_management.py:589-600; accumulate != 0 adds into stats_dev.  Deterministic. */
int imx_eval_len(const imx_env* env);   /* 4 + m */
int imx_eval_accumulate(imx_env* env, const void* obs_dev, const double* reward_dev, const double* profit_dev,
                        double* acc_dev, int reset, void* stream);
int imx_eval_stats(imx_env* env, const double* acc_dev, double* stats_dev, int accumulate, void* stream);

/* central_critic_observer + FillInActions  —  models/CC_Model.py:165-214 (and the hand-built CC
 * observation of CC_inv_management.py:516-528): for every agent the flat vector
 * [opponent_action (m-1) | opponent_obs (m-1)*O | own_obs O], W = imx_cc_obs_len() values.
 *   obs_dev      [N][m][O] in the element type this env writes (float64, or float32 with cfg.obs_f32)
 *   actions_dev  [N][m] float64 actions of the same step, clipped to [clip_lo, clip_hi]; NULL = zeros
 *   out_dev      [N][m][W] float64, or float32 when out_is_f32 != 0 (RLlib casts observations to float32) */
int imx_cc_obs_len(const imx_env* env);
int imx_cc_observe(imx_env* env, const void* obs_dev, const double* actions_dev, double clip_lo, double clip_hi,
                   void* out_dev, int out_is_f32, void* stream);

/* step(action) + central_critic_observer in ONE kernel: the step kernel's epilogue assembles the critic rows of
 * imx_cc_observe from the observation tile it has just built in shared memory and from this step's action tile, and
 * writes them with one bulk store per tile next to obs / reward / state (no second pass over [N][m][O]).
 *   obs_dev     [N][m][O] or NULL (the rows still contain every agent's observation)
 *   cc_dev      [N][m][W], W = imx_cc_obs_len(), in the observation element type (float64, or float32 with cfg.obs_f32)
 *   fill_actions non-zero: opponent-action slots = this step's actions clipped to [clip_lo, clip_hi] (FillInActions,
 *               models/CC_Model.py:165-193; the evaluation loops' hand-built rows, CC_inv_management.py:516-528); zero: zeros, as
 *               central_critic_observer leaves them at sampling time (:196-214)
 * Fused wherever the runtime-specialised TMA kernels serve the whole batch (N a multiple of the tile size, 16-byte aligned
 * buffers); otherwise imx_step followed by imx_cc_observe — same bytes either way.  Multi-agent kinds only. */
int imx_step_cc(imx_env* env, const double* actions_dev, void* obs_dev, void* cc_dev, int fill_actions, double clip_lo,
                double clip_hi, double* reward_dev, void* stream);

/* End-to-end convenience calls on HOST buffers (pinned memory recommended): copy in, launch, copy
 * out, synchronise.  These are what a per-step Python caller pays for. */
int imx_reset_host(imx_env* env, const int32_t* demand_host, const uint8_t* delay_mask_host, int noisy,
                   uint64_t episode, void* obs_host);
int imx_step_host(imx_env* env, const double* actions_host, void* obs_host, double* reward_host);

/* Poisson CDF table the Philox demand generator inverts (cdf[k] = P(X <= k), last entry a
 * sentinel > 1).  Returns the table length; copies min(len, cap) entries when out != NULL. */
int imx_poisson_cdf(const imx_env* env, double* out, int cap);

/* Which kernel served the last step()/rollout of this handle: 0 ahead-of-time direct kernel,
 * 1 ahead-of-time TMA-staged kernel, 2 runtime-specialised (NVRTC, same sources, flags as literals),
 * 3 runtime-specialised persistent pipeline (imx_step_pipe.cuh), 4 the one-launch episode kernel (imx_replay_episode). */
int imx_kernel_variant(const imx_env* env);
/* Last message of the runtime-specialisation layer (why it is unavailable, or a compile log). */
const char* imx_jit_log(void);
/* Compiles the specialised kernels for `cfg` with NVRTC for sm_100a WITHOUT a GPU (build check; also warms the on-disk
 * cubin cache).  variant: 0 = the step / step_many / rollout / pipelined kernels, 1 = the same without observations
 * (obs_dev = NULL), 2 = with the centralised-critic rows (imx_step_cc), 3 = imx_replay_episode's episode kernel,
 * 4 = the same without observations.
 * Returns the cubin size in bytes, or a negative error; `log` receives the compiler log. */
int imx_jit_compile_check(const imx_config* cfg, int variant, char* log, int cap);

/* Number of kernels this library has launched since load (bench.py's gpu_launches claim). */
int64_t imx_launch_count(void);
#endif /* !__CUDACC_RTC__ */

#ifdef __cplusplus
}
#endif
#endif /* IMX_B200_H */
