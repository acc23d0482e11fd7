/*
 * shems_b200.h — flat C ABI of libshems_b200.so (CUDA, sm_100a).
 *
 * This is the drop-in boundary for ONE hot path of RL-SHEMS: the batched
 * `shems_LU1` environment step/reset and the DDPG minibatch update.  The
 * reference has no FFI of its own (it is Julia multiple dispatch on the
 * Reinforce.jl protocol); every entry point below names the reference
 * function (file:line under /root/reference/RL-SHEMS/) it stands in for.  A
 * Julia maintainer binds these with `ccall((:sym, "libshems_b200"), Cint, …)`
 * — see INTEGRATION.md and the shim in <package>/julia/ShemsB200.jl.
 *
 * Conventions
 *   - Every function returns an int32 status: 0 = ok, <0 = error (enum below).
 *     A human-readable message for the last error on the calling thread is
 *     returned by shems_last_error().  Nothing throws or aborts across the ABI.
 *   - Handles are opaque; the library owns all device memory it allocates.
 *   - Pointers named *_dev are DEVICE pointers borrowed for the call (async:
 *     until the handle's stream is synchronised); pointers named *_host are
 *     host pointers, copied before return.
 *   - Batched arrays are structure-of-arrays: a "[k][N]" array stores field k
 *     of env n at offset k*N + n (coalesced over n).
 *   - A handle is not thread-safe; one handle <-> one CUDA stream.  Different
 *     handles may be used from different threads.
 *   - There is NO CPU fallback: on a box without a CUDA device every compute
 *     entry point fails with SHEMS_ERR_CUDA.
 */
#ifndef SHEMS_B200_H
#define SHEMS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SHEMS_API __attribute__((visibility("default")))

/* ------------------------------------------------------------------ status */
enum {
  SHEMS_OK = 0,
  SHEMS_ERR_INVALID = -1,  /* bad argument (NULL, size, range)                         */
  SHEMS_ERR_CUDA = -2,     /* CUDA runtime error, or no device                          */
  SHEMS_ERR_BOUNDS = -3,   /* row idx+1 > nrows: Julia BoundsError, shems_LU1.jl:266-268 */
  SHEMS_ERR_KEY = -4,      /* unknown charger id: Julia KeyError, shems_LU1.jl:95        */
  SHEMS_ERR_STATE = -5     /* call order (e.g. step before reset, sample from empty); a data-parallel gradient exchange that timed out */
};

SHEMS_API const char* shems_last_error(void);
SHEMS_API int32_t shems_version(void);
/* environment kernels (reset / step / action / rollout) this process has launched so far — a real counter for benchmarks' launch counts */
SHEMS_API int64_t shems_env_kernel_launches(void);
/* of those, rollouts that ran two instances per thread (all instances on one row; see DESIGN.md, rollout) */
SHEMS_API int64_t shems_rollout_pair_launches(void);
/* number of visible CUDA devices (0 on a CPU-only box; never an error) */
SHEMS_API int32_t shems_device_count(void);

/* ------------------------------------------------------------- environment */
#define SHEMS_STATE_SIZE 9   /* ShemsState, shems_LU1.jl:101-111 */
#define SHEMS_ACTION_SIZE 2  /* ShemsAction, shems_LU1.jl:146-149 */
#define SHEMS_TRACE_COLS 23  /* results row, shems_LU1.jl:476-478 */
#define SHEMS_SERIES_COLS 8

/* state field order (ShemsState, shems_LU1.jl:101-111) */
enum {
  SHEMS_S_SOC_B = 0, SHEMS_S_SOC_EV, SHEMS_S_C_EV, SHEMS_S_D_E, SHEMS_S_G_E,
  SHEMS_S_P_BUY, SHEMS_S_H_COS, SHEMS_S_H_SIN, SHEMS_S_SEASON
};

/* input-series columns the env reads (shems_LU1.jl:251-260, 268-279), in the
 * order of state fields 1..8.  Host layout handed to shems_create is
 * [SHEMS_SERIES_COLS][nrows] float32 (CSV Float64/Int values converted to
 * Float32 exactly as `env.state.x = df[idx, :col]` converts them). */
enum {
  SHEMS_COL_SOC_EV = 0,     /* :soc_ev        */
  SHEMS_COL_H_COUNTDOWN,    /* :h_countdown   */
  SHEMS_COL_ELECTKWH,       /* :electkwh      */
  SHEMS_COL_PV_GENERATION,  /* :PV_generation */
  SHEMS_COL_P_BUY,          /* :p_buy         */
  SHEMS_COL_HOUR_COS,       /* :hour_cos      */
  SHEMS_COL_HOUR_SIN,       /* :hour_sin      */
  SHEMS_COL_SEASON          /* :season        */
};

/* trace columns (shems_LU1.jl:476-478; CSV header memory_plotting_saving.jl:172-174) */
enum {
  SHEMS_T_INDEX = 0, SHEMS_T_C_EV, SHEMS_T_EV_TARGET, SHEMS_T_EV, SHEMS_T_SOC_EV,
  SHEMS_T_REWARD, SHEMS_T_PROFIT, SHEMS_T_DISCOMFORT, SHEMS_T_PENALTY, SHEMS_T_PV_DE,
  SHEMS_T_B_DE, SHEMS_T_GR_DE, SHEMS_T_PV_B, SHEMS_T_PV_GR, SHEMS_T_PV_EV, SHEMS_T_B_EV,
  SHEMS_T_GR_EV, SHEMS_T_EX_EV, SHEMS_T_GR_B, SHEMS_T_B_GR, SHEMS_T_B, SHEMS_T_B_TARGET,
  SHEMS_T_SOC_B
};

/* Module-level constants of shems_LU1.jl:40-43, 67-99 with their Julia types
 * (the Float64 fields matter: they drive the Float32->Float64 promotions). */
typedef struct ShemsParams {
  float pv_eta;                /* PV(1f0)                         :92  */
  float b_eta;                 /* Battery.eta = 0.95f0            :95  */
  float b_soc_min;             /* 0f0                             :95  */
  float b_soc_max;             /* capacities[id][2]               :47-59 */
  double b_rate_max;           /* capacities[id][3] (Float64)     :75  */
  float b_loss;                /* 0.00003f0                       :95  */
  float ev_soc_min;            /* 0f0                             :97  */
  float ev_soc_max;            /* capacities[id][1]               :47-59 */
  float ev_rate_max;           /* 11f0                            :97  */
  float penalty_weight;        /* 0.1f0                           :43  */
  double sell_discount;        /* Float64(0.2f0)                  :99, :86 */
  double discomfort_weight_ev; /* Float64(0.01f0)                 :40, :87 */
  double disc_pot;             /* Float64(2f0)                    :41, :88 */
  /* sibling environments (SURVEY §8 f4), all zero for shems_LU1: */
  double penalty_weight_f64;   /* `penalty_weight = 0.1` is a Float64 in shems_LU7.jl:35 and shems_LU1_input0607.jl:52, so
                                * `(1 - EV_target) * penalty_weight` is a Float64 product there (used when penalty_in_f64 != 0) */
  int32_t penalty_in_f64;
  int32_t reward_form;         /* 0: profit - w*discomfort^pot - penalty (shems_LU1.jl:467-470; shems_LU7.jl:465-468 with pot = 1)
                                * 1: profit - (discomfort*w)^pot - penalty (shems_LU1_input0607.jl:481-484) */
} ShemsParams;

/* capacities[charger_id] lookup (shems_LU1.jl:45-59, 92-99).  Unknown id ->
 * SHEMS_ERR_KEY (the reference raises KeyError at module load). */
SHEMS_API int32_t shems_params_for_charger(int32_t charger_id, ShemsParams* out);
/* the same for the sibling environment files of RL_environments/envs/ (module-level constants of each file):
 *   SHEMS_ENV_LU1            shems_LU1.jl (== shems_params_for_charger)
 *   SHEMS_ENV_LU7            shems_LU7.jl: battery 10 kWh / Float64(4.6f0) kW for every charger (:91), sell_discount 0.3f0, discomfort
 *                            weight 1 with a linear term (:94, :465-468), penalty_weight 0.1::Float64 (:35), EV capacities :42-55
 *   SHEMS_ENV_LU1_INPUT0607  shems_LU1_input0607.jl: (discomfort*w)^pot with pot = 1f0 (:49, :481-484), w = 0.1f0 (JOB digit 0; set
 *                            discomfort_weight_ev for the other grid-search alternatives :38-47), penalty_weight 0.1::Float64 (:52) */
enum { SHEMS_ENV_LU1 = 0, SHEMS_ENV_LU7 = 1, SHEMS_ENV_LU1_INPUT0607 = 2 };
SHEMS_API int32_t shems_params_for_env(int32_t env_variant, int32_t charger_id, ShemsParams* out);

/* CSV.read(env.path, DataFrame) (shems_LU1.jl:217, :265) done ONCE: parses `data/ChargerXX_all_{train,eval,test}_fix.csv` by column
 * name (21-column schema of Data_preparation_v2.ipynb cell 35) into the [8][nrows] float32 layout shems_create takes.
 * series_out == NULL: only *nrows_out is set (call again with a [8][capacity] buffer, capacity >= that row count; column k
 * then starts at series_out + k*capacity).  A missing column -> SHEMS_ERR_KEY; unreadable file / field -> SHEMS_ERR_INVALID. */
SHEMS_API int32_t shems_series_from_csv(const char* path, float* series_out, int32_t capacity, int32_t* nrows_out);

typedef struct ShemsEnv ShemsEnv; /* N instances of `Shems` (shems_LU1.jl:169-177) */

/* Shems(maxsteps, path) for n_envs instances (shems_LU1.jl:203) — the series
 * is parsed ONCE by the caller and uploaded here (the reference re-parses the
 * CSV at :217 and :265 on every reset/step).  device = CUDA ordinal. */
SHEMS_API int32_t shems_create(const ShemsParams* params, const float* series_host,
                               int32_t nrows, int32_t maxsteps, int64_t n_envs,
                               int32_t device, ShemsEnv** out);
/* The same for n_groups (<= 16) groups of instances: group g = group_sizes[g] consecutive instances with the constants params[g]
 * (one charger each, shems_LU1.jl:45-59) and, when series_per_group != 0, its own series (series_host [G][8][nrows], else
 * [8][nrows] shared).  The reference needs one Julia process per charger (JOB_ID digits, shems_LU1.jl:17,45). */
SHEMS_API int32_t shems_create_groups(const ShemsParams* params, int32_t n_groups, const int64_t* group_sizes, const float* series_host,
                                      int32_t series_per_group, int32_t nrows, int32_t maxsteps, int32_t device, ShemsEnv** out);
SHEMS_API int32_t shems_destroy(ShemsEnv* env);
/* use an existing CUDA stream (cudaStream_t) for all launches of this handle */
SHEMS_API int32_t shems_set_stream(ShemsEnv* env, void* cuda_stream);
SHEMS_API int32_t shems_sync(ShemsEnv* env);

/* reset!(env; rng) for all instances (shems_LU1.jl:206-262).
 *   mode SHEMS_RESET_DETERMINISTIC  == `rng == -1`: idx = 1, Soc_b = 0.5*(soc_min+soc_max).
 *   mode SHEMS_RESET_HOST_DRAWS     : the caller supplies the two draws the reference
 *        takes from MersenneTwister(rng) (:224-225): idx0_host[n] in 1..nrows-maxsteps and
 *        socb0_host[n]; the window-shift loop (:227-246) runs on the device.
 *   mode SHEMS_RESET_DEVICE_PHILOX  : draws come from Philox4x32-10 keyed by (seed, global
 *        env id) — Julia's MersenneTwister stream is not reproduced.
 * env_id_base offsets the global env id (multi-GPU sharding: results do not depend on the
 * number of ranks). */
enum { SHEMS_RESET_DETERMINISTIC = 0, SHEMS_RESET_HOST_DRAWS = 1, SHEMS_RESET_DEVICE_PHILOX = 2 };
SHEMS_API int32_t shems_reset(ShemsEnv* env, int32_t mode, const int32_t* idx0_host,
                              const float* socb0_host, uint64_t seed, int64_t env_id_base);

/* step!(env, s, a; track) for all instances (shems_LU1.jl:343-485).
 *   act_dev   [2][N] float: track >= 0 -> (B_target, EV_target) in [0,1]; track < 0 -> (B, EV) kWh.
 *   track     0 learning, 1 DRL inference, <0 rule-based bookkeeping (only the sign is used, :346-354, :466-471).
 *   reward_dev[N] float or NULL: Float32(env.reward) (what `cu` makes of the memory's rewards, memory_plotting_saving.jl:37).
 *   reward64_dev[N] double or NULL: env.reward::Float64 (:171, :467-470) — what episode! sums into reward_eps (DDPG.jl:223).
 *   obs_dev   [9][N] float or NULL: Vector{Float32}(env.state) after the step (NULL: read it
 *             later through shems_state_ptr — the handle's own state IS that array).
 *   trace_dev [23][N] double or NULL: the `results` row (:476-478).
 * Fails with SHEMS_ERR_BOUNDS (nothing launched) when any instance would read row idx+1 > nrows. */
SHEMS_API int32_t shems_step(ShemsEnv* env, const float* act_dev, int32_t track,
                             float* reward_dev, double* reward64_dev, float* obs_dev, double* trace_dev);

/* action(env, track) — the rule-based controller (shems_LU1.jl:318-340) -> (B, EV) [2][N] */
SHEMS_API int32_t shems_action_rule(ShemsEnv* env, float* bev_dev);
/* action(env, a::ShemsAction) (shems_LU1.jl:283-316): targets [2][N] -> feasible (B, EV) [2][N] */
SHEMS_API int32_t shems_action_drl(ShemsEnv* env, const float* target_dev, float* bev_dev);
/* finished(env, s') (shems_LU1.jl:487-502): always 0, kept for API completeness */
SHEMS_API int32_t shems_finished(const ShemsEnv* env, int32_t* out);

/* env.state / env.idx / env.step accessors (shems_LU1.jl:169-177) */
SHEMS_API int32_t shems_state_ptr(ShemsEnv* env, float** obs_dev /* [9][N] */, int32_t** idx_dev /* [N], 1-based */);
SHEMS_API int32_t shems_get_state(ShemsEnv* env, float* obs_host /* [9][N] */, int32_t* idx_host /* [N] or NULL */);
SHEMS_API int32_t shems_set_state(ShemsEnv* env, const float* obs_host /* [9][N] */, const int32_t* idx_host /* [N] */);
SHEMS_API int32_t shems_get_step(const ShemsEnv* env, int32_t* step);
SHEMS_API int64_t shems_num_envs(const ShemsEnv* env);
SHEMS_API int32_t shems_num_rows(const ShemsEnv* env); /* nrow(df) of the series (shems_LU1.jl:225) */

/* Fused T-step rollout: episode!/populate_memory/inference loops with the policy evaluated
 * on the device (DDPG.jl:186-242, memory_plotting_saving.jl:9-29, 62-89).  State stays in
 * registers for T steps; what is written per step is chosen by the sink pointers. */
enum {
  SHEMS_POLICY_RULE = 0,    /* a = action(env, track); step!(env, s, a, track=-0.5)  (DDPG.jl:209-212) */
  SHEMS_POLICY_RANDOM = 1,  /* a = 2U-1 (stored), scaled to [0,1]^2, track=0        (memory_plotting_saving.jl:14-21) */
  SHEMS_POLICY_TAPE = 2     /* targets read from tape_dev [T][2][N], track=0: scaled to [0,1] (tape_unscaled = 0) or the unscaled
                             * actions in [-1,1] that remember() stores, scale_action applied on the device (tape_unscaled = 1; the
                             * only form allowed together with a replay sink) */
};
typedef struct ShemsReplay ShemsReplay;
typedef struct ShemsRolloutArgs {
  int32_t policy;
  int32_t n_steps;            /* T */
  uint64_t seed;              /* Philox key for SHEMS_POLICY_RANDOM */
  int64_t env_id_base;        /* global env id offset (sharding) */
  const float* tape_dev;      /* [T][2][N] or NULL */
  double* ep_return_dev;      /* [N] sum of rewards (Float64, DDPG.jl:223) or NULL */
  ShemsReplay* replay;        /* push (s, a, r, s', done=0) per env-step or NULL */
  double* trace_dev;          /* [T][23][N] or NULL */
  float* obs_traj_dev;        /* [T][9][N] post-step observations or NULL */
  float* reward_traj_dev;     /* [T][N] or NULL */
  int32_t tape_unscaled;      /* SHEMS_POLICY_TAPE: 1 = the tape holds a in [-1,1] (DDPG.jl:229), scaled by scale_action (:178-184) */
} ShemsRolloutArgs;
SHEMS_API int32_t shems_rollout(ShemsEnv* env, const ShemsRolloutArgs* args);

/* ----------------------------------------------------------- replay memory */
/* memory = CircularBuffer{Any}(MEM_SIZE) of [s, a, r, s', done] (input.jl:140,
 * memory_plotting_saving.jl:46-47), device-resident SoA ring. */
SHEMS_API int32_t replay_create(int64_t capacity, int32_t device, ShemsReplay** out);
SHEMS_API int32_t replay_destroy(ShemsReplay* rp);
SHEMS_API int32_t replay_set_stream(ShemsReplay* rp, void* cuda_stream);
SHEMS_API int64_t replay_length(const ShemsReplay* rp);
SHEMS_API int64_t replay_capacity(const ShemsReplay* rp);
/* physical slot the next push writes (a full memory's oldest record sits there): checkpoints of a memory with priorities restore
 * the same slot order, which the tree's sums follow */
SHEMS_API int64_t replay_head(const ShemsReplay* rp);
/* number of env series the ring holds copies of: a rollout from a series-consistent env stores 32-byte compact records that
 * name a row of such a copy instead of the 88-byte transition (SHEMS_RING_COMPACT=0 forces full records) */
SHEMS_API int32_t replay_series_count(const ShemsReplay* rp);
/* remember(s, a, r, s', done) for n transitions (memory_plotting_saving.jl:46-47);
 * a is the UNSCALED action in [-1,1] (DDPG.jl:229). done_dev may be NULL (finished == false). */
SHEMS_API int32_t replay_push(ShemsReplay* rp, const float* s_dev /*[9][n]*/, const float* a_dev /*[2][n]*/,
                              const float* r_dev /*[n]*/, const float* s2_dev /*[9][n]*/,
                              const float* done_dev /*[n] or NULL*/, int64_t n);
/* remember() for a population of learners in one launch: the arrays are structure-of-arrays over all N = n_groups*n_per instances
 * ([9][N], [2][N], [N]; what an environment handle with N instances produces); learner l = instances l*n_per .. l*n_per+n_per-1
 * pushes its n_per transitions into rps[l].  All memories must live on one device; rps[0]'s stream is used. */
SHEMS_API int32_t replay_push_groups(ShemsReplay* const* rps, int32_t n_groups, const float* s_dev, const float* a_dev, const float* r_dev,
                                     const float* s2_dev, const float* done_dev, int64_t n_per);
/* getData(batch) (memory_plotting_saving.jl:31-42): i.i.d. WITH replacement.
 * idx_host != NULL: the caller's 0-based logical indices (0 = oldest), else Philox(seed).
 * Outputs are device arrays [9][B], [2][B], [B], [9][B], [B]. */
SHEMS_API int32_t replay_sample(ShemsReplay* rp, int32_t batch, const int32_t* idx_host, uint64_t seed,
                                float* s_dev, float* a_dev, float* r_dev, float* s2_dev, float* done_dev);
/* Proportional prioritized replay (Schaul et al., 2016; no reference counterpart).  replay_enable_priorities gives the memory a sum
 * tree of per-slot priorities: every filled slot gets p_max (which starts at 1), and from then on every slot a writer fills
 * (replay_push, replay_push_groups, shems_rollout with this replay, ddpg_episode) gets the p_max current in stream order.  Internal
 * nodes are always RN32(left + right) of their children.  A memory without priorities pays nothing. */
SHEMS_API int32_t replay_enable_priorities(ShemsReplay* rp);
/* priorities of the len records in logical order (0 = oldest) and p_max; synchronises the memory's stream.  SHEMS_ERR_STATE
 * without priorities. */
SHEMS_API int32_t replay_get_priorities(ShemsReplay* rp, float* prio_host /*[len]*/, float* p_max);
/* checkpoint restore: the len priorities in logical order and p_max, then the whole tree is recomputed.  Priorities must be finite
 * and >= 0 with at least one > 0, p_max finite and > 0; else SHEMS_ERR_INVALID and nothing changes. */
SHEMS_API int32_t replay_set_priorities(ShemsReplay* rp, const float* prio_host /*[len]*/, float p_max);
/* what update 0 of ddpg_update(seed) on a prioritized learner draws and weighs, enqueued on the memory's stream: draw j is
 * U = u53(Philox(seed, j, 0, STREAM_PER)), x = RN32((j + U) root / batch), then down the tree (left if x < L or R == 0, else
 * x = RN32(x - L) and right); idx_dev[j] = its logical index; w_dev[j] = RN32(x_j^-beta / max_k x_k^-beta) with
 * x_j = leaf_j len / root in Float64.  batch <= the memory's length is not required (draws are with replacement). */
SHEMS_API int32_t replay_sample_prioritized(ShemsReplay* rp, int32_t batch, uint64_t seed, float beta, int32_t* idx_dev /*[batch]*/,
                                            float* w_dev /*[batch]*/);
/* n-step returns (no reference counterpart).  replay_enable_successors gives the memory a successor link per slot, and every
 * existing record starts with none.  After every write (replay_push: one step of n instances; replay_push_groups: n_per; shems_rollout
 * with this replay: n_envs; ddpg_episode: the instances of its learner), in stream order, each new record i gets no successor, and the
 * record W before it (W the write's instances per step), if it has done == 0 and its s' equals s(i) in all 9 fields bit for bit, gets
 * i as its successor.  Episode boundaries end a chain by themselves (a reset breaks the equality).  A memory without links pays
 * nothing. */
SHEMS_API int32_t replay_enable_successors(ShemsReplay* rp);
/* successor of each of the len records in logical order (0 = oldest): a logical index, or -1; synchronises the memory's stream.
 * SHEMS_ERR_STATE without links. */
SHEMS_API int32_t replay_get_successors(ShemsReplay* rp, int32_t* next_host /*[len]*/);
/* checkpoint restore: the len successors in logical order; each must be -1 or in (i, len), else SHEMS_ERR_INVALID and nothing
 * changes.  SHEMS_ERR_STATE without links. */
SHEMS_API int32_t replay_set_successors(ShemsReplay* rp, const int32_t* next_host /*[len]*/);
/* what update 0 of ddpg_update(seed) trains on for an n-step learner with discount gamma, enqueued on the memory's stream: row j
 * starts at the record ring_draw(seed, j) picks (or idx_host[j], a logical index) and walks its successors in Float64 with explicit
 * roundings: gp = 1, R = r_0, k = 1; while k < n, done_{k-1} == 0 and the record has a successor: gp = RN64(gp gamma),
 * R = RN64(R + RN64(gp r_k)), k += 1.  s, a: the first record's; s2: the last record's s'; r = RN32(R);
 * done = RN32(1 - RN64(gp RN64(1 - done_{k-1}))), so the 1-step target r + gamma (1 - done) q' bootstraps with gamma^k; k_dev[j] = k
 * (k_dev may be NULL).  1 <= n <= 16, gamma in [0, 1]; n > 1 needs links (SHEMS_ERR_STATE). */
SHEMS_API int32_t replay_sample_nstep(ShemsReplay* rp, int32_t batch, const int32_t* idx_host, uint64_t seed, int32_t n, float gamma,
                                      float* s_dev, float* a_dev, float* r_dev, float* s2_dev, float* done_dev, int32_t* k_dev);
/* min_max_buffer(n) (memory_plotting_saving.jl:50-53): min/max of s over a with-replacement
 * sample of size n_samples -> s_min_host[9], s_max_host[9]. */
SHEMS_API int32_t replay_minmax(ShemsReplay* rp, int64_t n_samples, const int32_t* idx_host, uint64_t seed,
                                float* s_min_host, float* s_max_host);
/* host copies for tests / checkpoints: logical order, oldest first; arrays [k][len] */
SHEMS_API int32_t replay_get(ShemsReplay* rp, float* s_host, float* a_host, float* r_host,
                             float* s2_host, float* done_host);

/* ----------------------------------------------------------- DDPG learner */
typedef struct DdpgParams {
  int32_t state_size;   /* STATE_SIZE = 9            input.jl:180 */
  int32_t action_size;  /* ACTION_SIZE = 2           input.jl:181 */
  int32_t l1, l2;       /* L1, L2 (250, 500 tuned)   README.md:68-86 */
  int32_t batch;        /* BATCH_SIZE (120 tuned)    */
  float gamma;          /* γ   DDPG.jl:133 */
  float tau;            /* τ   DDPG.jl:142-143 */
  float lr_actor;       /* η_act,  ADAM(η_act)   input.jl:126-127 */
  float lr_critic;      /* η_crit, ADAM(η_crit) */
  double adam_beta1;    /* 0.9   (Flux.ADAM default) */
  double adam_beta2;    /* 0.999 */
  double adam_eps;      /* 1e-8  (Flux 0.12.1 const ϵ) */
  float act_lo[2];      /* ACTION_BOUND_LO input.jl:183 */
  float act_hi[2];      /* ACTION_BOUND_HI input.jl:182 */
  int32_t use_tensor_cores; /* 0: fp32 SIMT GEMMs (parity path); 1: TF32 tensor cores where the batch allows */
  int32_t population;       /* 0/1: the reference's single learner; P > 1: P independent learners (own nets, optimisers, replay
                             * memory, seeds) advanced by the same launches — BASELINE configs[4], the reference's one-process-per-seed
                             * parallelism (RL-SHEMS_bs_scheduler_*.sh:73-81) folded into one handle */
} DdpgParams;

/* DDPG_NET_ACTOR_BEST: the best-actor slot of a learner (what ddpg_keep_best keeps; ddpg_evaluate can run it).  ddpg_get_layer,
 * ddpg_set_layer and ddpg_num_params accept it; every other call that takes a net rejects it with SHEMS_ERR_INVALID. */
enum { DDPG_NET_ACTOR = 0, DDPG_NET_CRITIC = 1, DDPG_NET_ACTOR_TARGET = 2, DDPG_NET_CRITIC_TARGET = 3, DDPG_NET_ACTOR_BEST = 4 };

typedef struct Ddpg Ddpg;
SHEMS_API int32_t ddpg_default_params(DdpgParams* out);
/* builds actor/critic and their targets (DDPG.jl:30-46) with zero weights; call ddpg_init or ddpg_set_params */
SHEMS_API int32_t ddpg_create(const DdpgParams* p, int32_t device, Ddpg** out);
SHEMS_API int32_t ddpg_destroy(Ddpg* h);
SHEMS_API int32_t ddpg_set_stream(Ddpg* h, void* cuda_stream);
SHEMS_API int32_t ddpg_sync(Ddpg* h);
/* One learner at a small batch (batch % 8 == 0, batch <= 256, l1 <= 256, l2 <= 512, no tensor-core mode — the reference's B = 120,
 * 250/500 of README.md:68-86) runs replay() (DDPG.jl:121-145) as two thread-block-cluster kernels that keep every minibatch row's
 * forward/backward chain in shared memory (csrc/ddpg_fused.cu) instead of one launch per matrix product.  On by default where the
 * shape allows (environment variable SHEMS_DDPG_FUSED=0 opts out at ddpg_create); on = 0 selects the tiled-GEMM sequence (the
 * path populations, large batches and the data-parallel learner use).  Both are fp32 and deterministic; they differ by summation
 * order.  Returns the resulting state (1 fused, 0 not) or a negative status. */
SHEMS_API int32_t ddpg_set_fused(Ddpg* h, int32_t on);
/* Prioritized replay for every learner of the handle (on != 0) or uniform draws (on = 0, the default).  A prioritized update draws
 * its minibatch from the memory's sum tree (replay_sample_prioritized), scales the critic's output gradient of row j by its
 * importance weight (dq_j = RN32(dq_j w_j); the reported critic loss stays the unweighted mse) and writes the priority
 * p_j = RN32((|RN32(y_j - q_j)| + eps)^alpha) back to the slot it drew (a slot drawn twice takes the larger), p_max = max(p_max, p_j).
 * Caller-supplied indices (idx_host) are weighed and written back the same way.  Its updates take the tiled-GEMM sequence, never the
 * cluster-fused passes; act(), ddpg_rollout and ddpg_evaluate are unchanged.  alpha >= 0, beta in [0, 1], eps > 0, all finite, else
 * SHEMS_ERR_INVALID and nothing changes (the values are ignored for on = 0).  alpha, beta, eps are handle-wide and written in
 * stream order like ddpg_set_hparams (a beta schedule needs no re-capture).  Every update and training episode then needs memories
 * with priorities, one per learner (else SHEMS_ERR_STATE / SHEMS_ERR_INVALID, nothing launched); ddpg_update_batch,
 * ddpg_update_phase, ddpg_dp_connect and ddpg_update_dp return SHEMS_ERR_STATE on a prioritized handle. */
SHEMS_API int32_t ddpg_set_prioritized(Ddpg* h, int32_t on, float alpha, float beta, float eps);
SHEMS_API int32_t ddpg_get_prioritized(Ddpg* h, int32_t* on, float* alpha, float* beta, float* eps);
/* n-step returns for every learner of the handle (1 <= n <= 16; n = 1, the default, is the 1-step update).  With n > 1 each row of
 * an update from the replay memories is the walk replay_sample_nstep describes, with the learner's own gamma, and the unchanged TD
 * target r + gamma (1 - done) q' then is the n-step target.  The fused, tiled, tensor-core, chain and population paths all take it,
 * with uniform and with prioritized draws (a prioritized learner's priorities go back to the rows' first records).  n is handle-wide
 * and written in stream order (n > 1 to another n > 1 needs no re-capture).  Every update and training episode then needs memories
 * with links (replay_enable_successors, else SHEMS_ERR_STATE, nothing launched); ddpg_update_phase, ddpg_dp_connect and
 * ddpg_update_dp return SHEMS_ERR_STATE on an n-step handle, and so does n > 1 on a connected data-parallel learner.
 * ddpg_update_batch trains on the caller's minibatch as it is. */
SHEMS_API int32_t ddpg_set_nstep(Ddpg* h, int32_t n);
SHEMS_API int32_t ddpg_get_nstep(const Ddpg* h);
/* glorot_uniform hidden layers, U(-3e-3,3e-3) last layers, zero biases, targets = copies
 * (DDPG.jl:21-22, 30-46) from Philox(seed) (Julia's MersenneTwister stream is not reproduced); fresh optimisers
 * (ADAM moments zero, βp = β, update counter 0: input.jl:126-127). */
SHEMS_API int32_t ddpg_init(Ddpg* h, uint64_t seed);
/* Flux layout: layer weight is out×in column-major (element (o,i) at o + out*i), bias[out].
 * layer in 0..2.  Setting ACTOR/CRITIC does not touch the targets. */
SHEMS_API int32_t ddpg_set_layer(Ddpg* h, int32_t net, int32_t layer, const float* w_host, const float* b_host);
SHEMS_API int32_t ddpg_get_layer(Ddpg* h, int32_t net, int32_t layer, float* w_host, float* b_host);
SHEMS_API int64_t ddpg_num_params(const Ddpg* h, int32_t net);
/* s_min, s_max of normalize() (memory_plotting_saving.jl:55-57; frozen after driver:30) */
SHEMS_API int32_t ddpg_set_norm(Ddpg* h, const float* s_min_host, const float* s_max_host);
/* act(normalize(s); train) + scale_action (DDPG.jl:148-184) for n states:
 *   obs_dev [9][n] raw states; a_dev [2][n] clamp(actor(s_n)+noise,-1,1); scaled_dev [2][n] or NULL.
 *   noise_dev [2][n]: caller-provided noise (added as is) or NULL -> sigma*N(0,1) from Philox(seed, step)
 *   when sigma > 0 (GNoise, DDPG.jl:57-61), no noise when sigma == 0 (train == false). */
SHEMS_API int32_t ddpg_act(Ddpg* h, const float* obs_dev, int64_t n, float sigma, uint64_t seed, int64_t step,
                           int64_t env_id_base, const float* noise_dev, float* a_dev, float* scaled_dev);
/* ddpg_act with every array laid out as ONE structure-of-arrays over all N = P*n instances of a population (learner l owns
 * instances l*n .. l*n+n-1): obs_dev [9][N] is the state array of an environment handle (shems_state_ptr), scaled_dev [2][N] the
 * action array shems_step takes, noise_dev / a_dev [2][N].  For P == 1 it equals ddpg_act. */
SHEMS_API int32_t ddpg_act_soa(Ddpg* h, const float* obs_dev, int64_t n, float sigma, uint64_t seed, int64_t step, int64_t env_id_base,
                               const float* noise_dev, float* a_dev, float* scaled_dev);
/* act() with Ornstein-Uhlenbeck exploration noise (noise_type == "ou": sample_noise(ou::OUNoise) DDPG.jl:49-55, :157-158;
 * OUNoise(μ, σ, θ, dt, X) input.jl:190-234).  ou_x_dev [2][n] is OUNoise.X of every instance, read and advanced in place
 * (the reference never resets it, not even between episodes); z_dev [2][n]: the standard normal draws randn(2) (Float64)
 * or NULL -> Philox(seed, global env id, step) + Box-Muller.  Population handles: arrays gain a leading [P] dimension. */
SHEMS_API int32_t ddpg_act_ou(Ddpg* h, const float* obs_dev, int64_t n, float theta, float mu, float sigma, float dt, float* ou_x_dev,
                              uint64_t seed, int64_t step, int64_t env_id_base, const double* z_dev, float* a_dev, float* scaled_dev);
/* noise_type for ddpg_episode (input.jl:111): kind 0 = "gn" (default; sigma is passed per episode), 1 = "ou" with OUNoise(mu, sigma,
 * theta, dt, X) (input.jl:190-234); X is kept in the handle per instance and, like the reference's global `ou`, never reset. */
SHEMS_API int32_t ddpg_set_noise(Ddpg* h, int32_t kind, float theta, float mu, float dt);
/* episode!(env; NUM_STEPS, train, track = 0, rng_ep) (DDPG.jl:186-242) for every instance of `env`, enqueued by ONE call with no host
 * round trip per step: act(normalize(s)) (+ GNoise when train) -> scale_action -> step! -> remember -> replay() x updates_per_step.
 * reset! (:189) stays with the caller.  env holds N = P*n instances: learner l owns instances l*n .. l*n+n-1 and the memory rps[l]
 * (P = 1: the reference's loop).  Seeds: rng_step = (seed*1000003 + step) mod 2^63 keys the noise (with the global env id) and, as
 * rng_step + l, learner l's minibatch draws.  ep_return_dev [N] (Float64, or NULL) receives reward_eps (:223), noise_eps_dev [N]
 * (Float32, or NULL) noise_eps = the sum over the steps of mean(noise) (:224; what run_episodes stores in noise_mean).  The three handles
 * must share one CUDA stream; the call returns as soon as the work is enqueued.  On a handle connected with ddpg_dp_connect every
 * replay() is the data-parallel one (ddpg_update_dp: all ranks must make the same calls), so the replicas stay identical. */
SHEMS_API int32_t ddpg_episode(Ddpg* h, ShemsEnv* env, ShemsReplay* const* rps, int32_t n_steps, int32_t train, float sigma, uint64_t seed,
                               int32_t updates_per_step, int64_t env_id_base, double* ep_return_dev, float* noise_eps_dev);
/* episode!(env; NUM_STEPS, train = false, track, rng_ep) (DDPG.jl:186-242) and inference(env; track = 1) (memory_plotting_saving.jl:62-89,
 * 1439 / 2999 / 4319 steps from reset!(rng = -1)) for every instance of `env`, by ONE call: act(normalize(s)) [+ GNoise when
 * sigma > 0] -> scale_action -> step!, n_steps times.  One learner at widths l1 <= 256, l2 <= 512 runs as a single persistent
 * thread-block-cluster kernel (csrc/actor_rollout.cu: the actor's W2 stays in shared memory for the whole episode, 8 instances per
 * cluster, no launch and no host round trip per step); populations and wider nets take one act + step! launch pair per step.
 * The 100 evaluation episodes of run_episodes (DDPG.jl:266-279) are one call on an environment handle with 100 instances.
 *   ep_return_dev [N] double or NULL: reward_eps (:223);  trace_dev [T][23][N] double or NULL: the `results` rows of track = 1
 *   (:207-208);  act_traj_dev [T][2][N] float or NULL: the unscaled actions a.  Seeds as ddpg_episode; reset! stays with the caller. */
SHEMS_API int32_t ddpg_rollout(Ddpg* h, ShemsEnv* env, int32_t n_steps, float sigma, uint64_t seed, int64_t env_id_base,
                               double* ep_return_dev, double* trace_dev, float* act_traj_dev);
/* Evaluation and best-actor bookkeeping of run_episodes (DDPG.jl:266-289) for EVERY learner of the handle (P = 1 included).
 * ddpg_evaluate: episode!(env; train = false) / inference(env; track = 1) without noise, by ONE call: the persistent cluster kernel of
 * ddpg_rollout with a learner dimension (8 instances of one learner per cluster, that learner's actor and s_min / s_max), so a learner
 * evaluated inside a population gets the bits it gets on a one-learner handle.  net = DDPG_NET_ACTOR or DDPG_NET_ACTOR_BEST; env holds
 * N = P*n instances, learner l owns l*n .. l*n+n-1, and for P > 1 no group boundary of env may split a learner's instances.  Outputs, env_id_base,
 * preconditions (one stream, reset! first) and SHEMS_ERR_BOUNDS (nothing launched) as ddpg_rollout; SHEMS_ERR_INVALID also when l1 > 256
 * or l2 > 512 or a group splits a learner of a population.  For P == 1 and net = ACTOR it equals ddpg_rollout with sigma = 0. */
SHEMS_API int32_t ddpg_evaluate(Ddpg* h, ShemsEnv* env, int32_t net, int32_t n_steps, int64_t env_id_base, double* ep_return_dev,
                                double* trace_dev, float* act_traj_dev);
/* ddpg_keep_best: one enqueue, no host round trip.  For every learner l: score_l = (sum over k of ep_return_dev[l*n + k]) / n, summed in
 * index order in Float64 (score_mean, :273) and written to score_dev [P] unless NULL; if score_l > best_score_l (strict: a tie or NaN
 * never wins, :282) best_score_l = score_l, best_run_l = episode and learner l's actor is copied into its DDPG_NET_ACTOR_BEST slot.
 * ddpg_create starts every learner at best_score = -100000, best_run = 0 and a zero best actor.  ddpg_get_best / ddpg_set_best move the
 * [P] arrays (set: checkpoint restore, the start of run_episodes; the best-actor weights go through ddpg_set_layer(ACTOR_BEST)). */
SHEMS_API int32_t ddpg_keep_best(Ddpg* h, const double* ep_return_dev, int64_t n, int32_t episode, double* score_dev);
SHEMS_API int32_t ddpg_get_best(Ddpg* h, double* best_score_host, int32_t* best_run_host);
SHEMS_API int32_t ddpg_set_best(Ddpg* h, const double* best_score_host, const int32_t* best_run_host);
/* Population-based training (no reference counterpart: the reference runs one process per grid point and its author picks the best
 * seeds afterwards).  ddpg_exploit: one enqueue, no host allocation, no synchronisation (it fits between ddpg_keep_best and the next
 * ddpg_episode).  Learners split into contiguous groups [group_start[g], group_start[g+1]) (n_groups = 0: one group of all P);
 * nothing crosses a group.  In a group of m learners: key_l = score_dev[l] with NaN as -inf, rank_l = position in descending key order
 * with ties to the lower index, k = floor(frac * m) in double.  Every learner d with rank_d >= m - k (the bottom set) draws
 * w[4] = Philox4x32-10(seed, id = d, ctr = round, stream = 0x5042) and takes as its source s the learner of rank
 * (uint32)(((uint64)w[0] * k) >> 32) (the top set rank < k; the two sets are disjoint).  From s to d are copied exactly what
 * ddpg_get_state / ddpg_set_state move: actor, critic, both targets, the four ADAM moment arrays, s_min / s_max, and the β powers
 * (with their reciprocals) of both optimisers.  d keeps its own Philox seed and update counter, its replay memory, its best-actor
 * slot, best_score / best_run, OU state, gradients and scratch; the handle-wide update counter is unchanged.  Then each
 * hyper-parameter j with bit j of keys set (0 lr_actor, 1 lr_critic, 2 gamma, 3 tau, 4 noise_scale) becomes RN32(value_s * f), f =
 * factor_hi if bit j of w[1] is set else factor_lo, gamma and tau then min(x, 1); the others are copied.  parent_dev [P] (or NULL)
 * receives s for a replaced learner and -1 for the others.  k = 0 or m = 1 changes nothing in that group; P = 1 is valid.
 * ddpg_get_hparams after the call synchronises and shows the device values.  SHEMS_ERR_INVALID, with nothing launched: NULL h,
 * score_dev or p, frac NaN or outside [0, 0.5], a factor not finite or <= 0, keys outside 0..31, n_groups outside 0..16, group
 * starts that do not begin at 0, increase strictly and end at P. */
#define DDPG_EXPLOIT_MAX_GROUPS 16
typedef struct DdpgExploitParams DdpgExploitParams;
struct DdpgExploitParams {
  double frac;                 /* share of each group replaced and share it is drawn from, [0, 0.5] */
  float factor_lo, factor_hi;  /* perturbation factors, finite and > 0 */
  int32_t keys;                /* bit j set: perturb hyper-parameter j (0 lr_actor, 1 lr_critic, 2 gamma, 3 tau, 4 noise_scale) */
  uint32_t round;              /* Philox counter: the evaluation round */
  uint64_t seed;
  int32_t n_groups;            /* 0: one group of all P learners */
  int32_t group_start[DDPG_EXPLOIT_MAX_GROUPS + 1];
};
SHEMS_API int32_t ddpg_exploit(Ddpg* h, const double* score_dev, const DdpgExploitParams* p, int32_t* parent_dev);
/* replay() (DDPG.jl:121-145) n_updates times: sample -> TD target -> critic step -> actor step
 * -> Polyak.  idx_host ([n_updates][batch], 0-based logical indices) or NULL -> Philox(seed, draw j, counter u = index of the
 * update inside this call): replay(rng_rpl = r) trains on the minibatch replay_sample(seed = r) returns, as getData(rng) is one
 * sample in both of its uses (memory_plotting_saving.jl:31-42). */
SHEMS_API int32_t ddpg_update(Ddpg* h, ShemsReplay* rp, int32_t n_updates, const int32_t* idx_host, uint64_t seed);
/* the same update on a caller-supplied minibatch (device, [9][B],[2][B],[B],[9][B],[B]) */
SHEMS_API int32_t ddpg_update_batch(Ddpg* h, const float* s_dev, const float* a_dev, const float* r_dev,
                                    const float* s2_dev, const float* done_dev);
/* Data-parallel learner (one process per GPU): the same replay() in three calls.  After phase 0 the critic part of the
 * flat gradient buffer (ddpg_grad_buffer, first ddpg_num_params(CRITIC) floats) is final on this rank, after phase 1 the
 * actor part; the caller all-reduces (sum) each part over the ranks (NCCL) and passes grad_scale = 1/world_size to the
 * next phase, which applies ADAM to the averaged gradient.  grad_scale is ignored by phase 0. */
SHEMS_API int32_t ddpg_update_phase(Ddpg* h, ShemsReplay* rp, int32_t phase, const int32_t* idx_host, uint64_t seed, float grad_scale);
/* Population handles (DdpgParams.population = P > 1).  Batched arrays gain a leading [P] dimension: ddpg_act takes
 * obs_dev [P][9][n], noise_dev [P][2][n] and fills a_dev / scaled_dev [P][2][n]; ddpg_init seeds learner l with seed + l;
 * get/set_layer, get_grad, set_norm and get_losses address the learner chosen by ddpg_select_learner (default 0).
 * ddpg_update_population: replay() n_updates times for every learner, learner l sampling rps[l] with Philox(seeds[l]) or
 * idx_host [P][n_updates][batch].  Also valid for P == 1 (ddpg_update is that case). */
SHEMS_API int32_t ddpg_select_learner(Ddpg* h, int32_t learner);
SHEMS_API int32_t ddpg_population(const Ddpg* h);
SHEMS_API int32_t ddpg_update_population(Ddpg* h, ShemsReplay* const* rps, int32_t n_updates, const int32_t* idx_host, const uint64_t* seeds);
/* Per-learner hyper-parameters of the learner chosen by ddpg_select_learner (valid for P == 1 too): the ADAM learning rates η_act,
 * η_crit, the discount γ, the Polyak rate τ and an exploration-noise scale.  ddpg_create gives every learner the DdpgParams values
 * and noise_scale = 1.  Wherever the library draws noise (ddpg_act*, ddpg_act_ou, ddpg_episode, ddpg_rollout) it uses
 * σ_eff = RN32(sigma × noise_scale) with the sigma of the call; caller-supplied noise_dev is added as is.  The write is ordered on
 * the handle's stream, so it applies to the next launch.  Values must be finite, lr_* >= 0, noise_scale >= 0 and gamma, tau in
 * [0, 1]; anything else returns SHEMS_ERR_INVALID and changes nothing.  Data-parallel ranks must all make the same call. */
SHEMS_API int32_t ddpg_set_hparams(Ddpg* h, float lr_actor, float lr_critic, float gamma, float tau, float noise_scale);
SHEMS_API int32_t ddpg_get_hparams(Ddpg* h, float* lr_actor, float* lr_critic, float* gamma, float* tau, float* noise_scale);
/* Data-parallel learner with the gradient all-reduce fused into the optimiser kernels over NVLink peer memory (one process per
 * GPU).  Each rank exports DDPG_DP_HANDLE_BYTES (the CUDA IPC handle of its exchange box: per-block flags and one inbound row of
 * gradient sums per peer, which the peers write), the caller gathers the
 * ranks' blobs in rank order (any transport: torch.distributed, MPI, a file) and hands them to ddpg_dp_connect.  ddpg_update_dp is
 * replay() with both exchanges done in-kernel: no NCCL call, no host synchronisation; all ranks must issue the same calls.
 * A peer that does not arrive within 4 s (environment SHEMS_DP_TIMEOUT_MS at connect time) makes the kernel give up without applying the
 * step (ddpg_dp_status reports 1, ddpg_sync fails) instead of hanging the GPU. */
#define DDPG_DP_HANDLE_BYTES 192
SHEMS_API int32_t ddpg_dp_export(Ddpg* h, void* handle_out /* [DDPG_DP_HANDLE_BYTES] */);
SHEMS_API int32_t ddpg_dp_connect(Ddpg* h, int32_t rank, int32_t world, const void* handles /* [world][DDPG_DP_HANDLE_BYTES] */);
/* optional: allocate/instantiate up front what ddpg_update_dp needs (idx_ints = n_updates*batch host indices per call, 0 if none) */
SHEMS_API int32_t ddpg_dp_prepare(Ddpg* h, int64_t idx_ints);
SHEMS_API int32_t ddpg_update_dp(Ddpg* h, ShemsReplay* rp, int32_t n_updates, const int32_t* idx_host, uint64_t seed);
SHEMS_API int32_t ddpg_dp_status(Ddpg* h, int32_t* error_out);
/* last update's loss_crit / loss_act values (DDPG.jl:114-119) */
SHEMS_API int32_t ddpg_get_losses(Ddpg* h, float* loss_crit, float* loss_act);
/* gradients of the last update (Flux layout, like ddpg_get_layer); net = ACTOR or CRITIC */
SHEMS_API int32_t ddpg_get_grad(Ddpg* h, int32_t net, int32_t layer, float* w_host, float* b_host);
/* flat fp32 gradient buffer on the device: critic gradient at [0, nc), actor gradient at [roundup(nc, 64), roundup(nc, 64) + na),
 * zero padding between them; *n = roundup(nc, 64) + na (nc, na = ddpg_num_params of critic / actor) */
SHEMS_API int32_t ddpg_grad_buffer(Ddpg* h, float** grad_dev, int64_t* n);

/* Full learner snapshot — what the reference never saves (saveBSON writes the actor and the score arrays only,
 * memory_plotting_saving.jl:263-270, so its runs cannot be resumed): of the learner chosen by ddpg_select_learner,
 *   state_host [ddpg_state_floats()] = [actor | critic | actor_target | critic_target | m_actor | v_actor | m_critic | v_critic |
 *                                       s_min (9) | s_max (9)]   (nets in the flat Flux layout of ddpg_get_layer, ADAM moments alike)
 *   opt_host [8] doubles             = [βp_critic[1], βp_critic[2], βp_actor[1], βp_actor[2] (Flux.ADAM's β^t), update counter, 0, 0, 0]
 * A learner restored with ddpg_set_state continues bit-identically (tests/test_resume_gpu.py); the replay memory is saved with
 * replay_get and restored with replay_push into a fresh memory of the same capacity (sampling uses logical indices). */
SHEMS_API int64_t ddpg_state_floats(const Ddpg* h);
SHEMS_API int32_t ddpg_get_state(Ddpg* h, float* state_host, double* opt_host);
SHEMS_API int32_t ddpg_set_state(Ddpg* h, const float* state_host, const double* opt_host);
/* OUNoise.X of ddpg_episode's instances ([2][n], input.jl:234; the reference never resets it): *n_out = instance count (0 before the
 * first OU episode), x_host may be NULL to query it; ddpg_set_ou_state (re)allocates for n instances. */
SHEMS_API int32_t ddpg_get_ou_state(Ddpg* h, float* x_host, int64_t* n_out);
SHEMS_API int32_t ddpg_set_ou_state(Ddpg* h, const float* x_host, int64_t n);

/* ------------------------------------------------ tensor-core GEMM (test / benchmark entry point)
 * The TF32 tcgen05 kernel behind the large-batch DDPG update, exposed for unit tests and roofline measurements:
 * D[M x N] (row-major, ldd) = epi(sum_k A(m,k) B(n,k)); *_mn = 0: operand is K-major ((row,k) at p[row*ld+k]),
 * 1: MN-major ((row,k) at p[k*ld+row]).  epi: 0 none, 1 bias+ReLU, 2 ReLU-mask by aux.  splits > 1: split-K through
 * workspace_dev (splits*M*N floats), reduced in a fixed order.  All pointers are device pointers, 16-byte aligned.  When ldd > N the
 * padding floats N .. roundup(N,4)-1 of a row may be overwritten with zeros (the tile store clips at 16 bytes); nothing beyond them. */
SHEMS_API int32_t shems_tc_gemm(const float* a_dev, int64_t lda, int32_t a_mn, const float* b_dev, int64_t ldb, int32_t b_mn,
                                float* d_dev, int64_t ldd, int32_t M, int32_t N, int32_t K, int32_t epi, const float* bias_dev,
                                const float* aux_dev, int64_t auxld, int32_t splits, float* workspace_dev, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* SHEMS_B200_H */
