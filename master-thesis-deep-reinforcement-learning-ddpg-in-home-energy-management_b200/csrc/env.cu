// env.cu — batched shems_LU1 environment: reset / step / actions / fused rollout kernels and
// their C-ABI entry points (include/shems_b200.h).  Compiled with -fmad=false (see shems_device.cuh).
//
// Data layout in HBM (per handle, N instances):
//   obs  [9][N] float   structure-of-arrays ShemsState; thread n touches obs[k*N + n] -> every
//                       access of a warp is one contiguous 128-byte line
//   idx  [N]    int32   env.idx (1-based row)
//   series [nrows] x 2 float4 = one 32-byte row per hour:
//                       (soc_ev, h_countdown, electkwh, PV_generation | p_buy, hour_cos, hour_sin, season)
//                       read-only, L1/L2 resident (<= 280 KB), fetched with ld.global.nc
#include <new>
#include <vector>
#include <string.h>
#include <math.h>
#include <stdlib.h>

#include "common.h"
#include "philox.cuh"
#include "shems_device.cuh"

// ----------------------------------------------------------------------------- errors
static thread_local char g_err[512] = "";
void shems_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
extern "C" const char* shems_last_error(void) { return g_err; }
extern "C" int32_t shems_version(void) { return 200; }
// environment kernels (reset / step / action / rollout) launched by this process so far: what bench.py reports as gpu_launches
static long long g_env_launches = 0;
extern "C" int64_t shems_env_kernel_launches(void) { return __atomic_load_n(&g_env_launches, __ATOMIC_RELAXED); }
#define COUNT_LAUNCH() __atomic_add_fetch(&g_env_launches, 1, __ATOMIC_RELAXED)
extern "C" int32_t shems_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

// ----------------------------------------------------------------------------- params
extern "C" int32_t shems_params_for_charger(int32_t charger_id, ShemsParams* p) {
  REQUIRE(p != nullptr, SHEMS_ERR_INVALID, "shems_params_for_charger: out is NULL");
  // capacities :: Dict{Int, Tuple{Float32, Float32, Float64}}  (shems_LU1.jl:47-59)
  struct Row { int id; float ev_cap, b_nom; double rate; };
  static const Row rows[] = {{1, 48.250f, 7.5f, 3.3},  {2, 36.271f, 10.f, 3.3}, {3, 45.508f, 10.f, 3.3}, {4, 78.993f, 11.f, 4.6},
                             {5, 37.207f, 10.f, 4.6},  {6, 35.816f, 15.f, 4.6}, {7, 36.521f, 12.f, 3.3}, {8, 45.728f, 10.f, 3.3},
                             {9, 21.935f, 7.5f, 3.3},  {98, 35.816f, 7.5f, 3.3}, {97, 78.993f, 11.f, 4.6}};
  for (const Row& r : rows) {
    if (r.id != charger_id) continue;
    p->pv_eta = 1.0f;
    p->b_eta = 0.95f;
    p->b_soc_min = 0.0f;
    { volatile float nom = r.b_nom, k = 0.9f; volatile float cap = nom * k; p->b_soc_max = cap; }  // `7.5f0 * 0.9f0`: one Float32 rounding
    p->b_rate_max = r.rate;
    p->b_loss = 0.00003f;
    p->ev_soc_min = 0.0f;
    p->ev_soc_max = r.ev_cap;
    p->ev_rate_max = 11.0f;
    p->penalty_weight = 0.1f;
    p->sell_discount = (double)0.2f;
    p->discomfort_weight_ev = (double)0.01f;
    p->disc_pot = 2.0;
    p->penalty_weight_f64 = 0.0; p->penalty_in_f64 = 0; p->reward_form = 0;
    return SHEMS_OK;
  }
  shems_set_error("KeyError: key %d not found in capacities (shems_LU1.jl:47-59)", charger_id);
  return SHEMS_ERR_KEY;
}

// module-level constants of the sibling environment files (SURVEY §8 f4)
extern "C" int32_t shems_params_for_env(int32_t env_variant, int32_t charger_id, ShemsParams* p) {
  REQUIRE(p != nullptr, SHEMS_ERR_INVALID, "shems_params_for_env: out is NULL");
  REQUIRE(env_variant >= SHEMS_ENV_LU1 && env_variant <= SHEMS_ENV_LU1_INPUT0607, SHEMS_ERR_INVALID, "shems_params_for_env: unknown variant %d", env_variant);
  if (env_variant == SHEMS_ENV_LU1) return shems_params_for_charger(charger_id, p);
  if (env_variant == SHEMS_ENV_LU1_INPUT0607) {
    // capacities as shems_LU1.jl without charger 97 (shems_LU1_input0607.jl:57-68)
    REQUIRE(charger_id != 97, SHEMS_ERR_KEY, "KeyError: key 97 not found in capacities (shems_LU1_input0607.jl:57-68)");
    const int32_t st = shems_params_for_charger(charger_id, p);
    if (st) return st;
    p->discomfort_weight_ev = (double)0.1f;  // fourth ternary digit 0 (:38-47)
    p->disc_pot = (double)1.0f;              // DISC_POT = 1f0 (:49)
    p->penalty_weight_f64 = 0.1; p->penalty_in_f64 = 1;  // penalty_weight = 0.1 (:52)
    p->reward_form = 1;                      // (discomfort * w)^pot (:481-484)
    return SHEMS_OK;
  }
  // shems_LU7.jl: ev_capacities :42-55 (ids 1-9, 98, 99), Battery(0.95f0, 0f0, 10f0, 4.6f0, 0.00003f0) :91, Market(0.3f0, 1) :94
  struct Row { int id; float ev_cap; };
  static const Row rows[] = {{1, 48.250f}, {2, 36.271f}, {3, 45.508f}, {4, 78.993f}, {5, 37.207f}, {6, 35.816f}, {7, 36.521f}, {8, 45.728f},
                             {9, 21.935f}, {99, 35.816f}, {98, 35.816f}};
  for (const Row& r : rows) {
    if (r.id != charger_id) continue;
    p->pv_eta = 1.0f; p->b_eta = 0.95f; p->b_soc_min = 0.0f; p->b_soc_max = 10.0f;
    p->b_rate_max = (double)4.6f;            // rate_max::Float64 <- 4.6f0
    p->b_loss = 0.00003f; p->ev_soc_min = 0.0f; p->ev_soc_max = r.ev_cap; p->ev_rate_max = 11.0f;
    p->penalty_weight = 0.1f;                // unused: the Float64 weight below is the one LU7 defines
    p->sell_discount = (double)0.3f;
    p->discomfort_weight_ev = 1.0;           // DISCOMFORT_WEIGHT_EV = 1 (Int -> Float64 field)
    p->disc_pot = 1.0;                       // linear term: discomfort * w == w * discomfort^1.0 exactly
    p->penalty_weight_f64 = 0.1; p->penalty_in_f64 = 1; p->reward_form = 0;
    return SHEMS_OK;
  }
  shems_set_error("KeyError: key %d not found in ev_capacities (shems_LU7.jl:42-55)", charger_id);
  return SHEMS_ERR_KEY;
}

// Exhaustive host check that q = x*r; e = fma(-q, d, x); q' = fma(e, r, q) equals the IEEE quotient x/d for every
// Float32 significand (the exponent of x only scales the computation while nothing is subnormal — the device falls back
// to the IEEE division below 2^-60).  ~10 ms per distinct divisor, cached.
static int verify_fdiv_const(float d) {
  static float cache_d[8]; static int cache_ok[8]; static int n_cache = 0;
  for (int i = 0; i < n_cache; ++i) if (memcmp(&cache_d[i], &d, 4) == 0) return cache_ok[i];
  int ok = (d == d) && d != 0.0f && fabsf(d) > 1e-30f && fabsf(d) < 1e30f;
  if (ok) {
    volatile float rv = 1.0f / d;
    const float r = rv;
    for (uint32_t m = 0x3f800000u; m < 0x40000000u && ok; ++m) {
      float x; memcpy(&x, &m, 4);
      volatile float q = x * r;
      const float e = fmaf(-q, d, x);
      const float q2 = fmaf(e, r, q);
      volatile float ref = x / d;
      if (q2 != ref) ok = 0;
    }
  }
  if (n_cache < 8) { cache_d[n_cache] = d; cache_ok[n_cache] = ok; ++n_cache; }
  return ok;
}

// RD32(c) / RU32(c): the Float32 neighbours of a Float64 c (c itself when it is Float32-valued); for Float32 x,
// x > c <=> x > RD32(c) and x < c <=> x < RU32(c)
static float f32_round_down(double c) {
  const float f = (float)c;
  return ((double)f > c) ? nextafterf(f, -INFINITY) : f;
}
static float f32_round_up(double c) {
  const float f = (float)c;
  return ((double)f < c) ? nextafterf(f, INFINITY) : f;
}

static DevParams make_dev_params(const ShemsParams& p) {
  DevParams d;
  d.pv_eta = p.pv_eta; d.b_eta = p.b_eta; d.smin = p.b_soc_min; d.smax = p.b_soc_max; d.loss = p.b_loss;
  d.evmin = p.ev_soc_min; d.evmax = p.ev_soc_max; d.evR = p.ev_rate_max; d.pw = p.penalty_weight;
  volatile float oml = 1.0f - p.b_loss;       // host fp32, rounded once (no x87, no contraction)
  volatile float omle = oml - 1e-7f;
  volatile float C = p.ev_soc_max - p.ev_soc_min;
  volatile float span = p.b_soc_max - p.b_soc_min;
  d.one_m_l = oml; d.one_m_l_e = omle; d.C = C; d.span = span;
  d.R_f = (float)p.b_rate_max;
  d.R = p.b_rate_max; d.sell = p.sell_discount; d.dw = p.discomfort_weight_ev; d.pot = p.disc_pot;
  d.pw_d = p.penalty_weight_f64; d.pen_f64 = p.penalty_in_f64 != 0; d.reward_form = p.reward_form != 0;
  d.reward_mode = (d.reward_form == 0 && p.disc_pot == 2.0) ? 0 : 1;
  d.eta_d = (double)p.b_eta; d.one_m_l_d = (double)d.one_m_l; d.C_d = (double)d.C;
  d.smax95 = 0.95 * (double)p.b_soc_max;
  { volatile float r1 = 1.0f / p.b_eta, r2 = 1.0f / d.span; d.r_eta_f = r1; d.r_span_f = r2; }
  d.r_eta_d = 1.0 / d.eta_d; d.r_C_d = 1.0 / d.C_d;
  d.fast_eta_f = verify_fdiv_const(p.b_eta);
  d.fast_span_f = verify_fdiv_const(d.span);
  // eta_d and C_d are converted Float32 values by construction (<= 24 significant bits): see ddiv_const
  d.fast_d = ((double)(float)d.eta_d == d.eta_d) && ((double)(float)d.C_d == d.C_d) && d.eta_d != 0.0 && d.C_d != 0.0;
  d.span_d = (double)d.span; d.r_span_d = 1.0 / d.span_d;
  d.R_dn = f32_round_down(d.R); d.R_up = f32_round_up(d.R); d.smax95_up = f32_round_up(d.smax95);
  d.fast_all = d.fast_d && d.span_d != 0.0 && d.span == d.span && fabs(d.span_d) < 1e30 && !d.pen_f64 && d.reward_mode == 0;
  return d;
}

// ----------------------------------------------------------------------------- reset
// reset!/reset_state! (shems_LU1.jl:206-262).  mode: SHEMS_RESET_*.
__global__ void __launch_bounds__(256)
shems_reset_kernel(DevParams P, const float4* __restrict__ series, int nrows, int maxsteps, long long N, int mode,
                   const int32_t* __restrict__ idx0_in, const float* __restrict__ socb0_in, unsigned long long seed,
                   long long env_id_base, float* __restrict__ obs, int32_t* __restrict__ idx_out, int32_t* __restrict__ maxidx,
                   long long n0, long long n1) {
  const long long n = n0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;  // this launch covers one group: instances n0 .. n1-1
  int idx = 1;
  if (n < n1) {
    const int hi = nrows - maxsteps;
    float Soc_b;
    if (mode == SHEMS_RESET_DETERMINISTIC) {  // rng == -1, :220-222
      Soc_b = (float)(0.5 * (double)(P.smin + P.smax));
      idx = 1;
    } else {
      int idx0;
      if (mode == SHEMS_RESET_HOST_DRAWS) {
        idx0 = idx0_in[n];
        Soc_b = socb0_in[n];
      } else {  // Philox draws standing in for the two MersenneTwister(rng) draws of :224-225
        uint32_t r[4];
        philox4x32_10(seed, (uint64_t)(env_id_base + n), 0u, STREAM_RESET, r);
        Soc_b = (float)((double)P.smin + (double)P.span * u53(r[0], r[1]));
        int k = (int)(u53(r[2], r[3]) * (double)hi);
        idx0 = 1 + (k >= hi ? hi - 1 : k);
      }
      idx = idx0;
      // :227-246 shift the window until it does not end inside a charging session
      float c_end = __ldg(&reinterpret_cast<const float*>(series)[8 * (size_t)(idx + maxsteps - 1) + 1]);
      int counter = 0;
      while (c_end > -1.0f && idx < hi) {
        idx += (int)(c_end + 1.0f);
        if (idx > hi) idx = idx0;  // the re-draw at :236 re-seeds MersenneTwister(rng): same index again
        c_end = __ldg(&reinterpret_cast<const float*>(series)[8 * (size_t)(idx + maxsteps - 1) + 1]);
        if (++counter > 100) break;  // :242-245
      }
    }
    const Row8 r = load_row(series, idx);  // :251-260
    store_obs(obs, N, n, Soc_b, r.soc_ev, r);
    idx_out[n] = idx;
  }
  // max idx of the block -> one atomic (bounds pre-check of the following steps)
  int m = idx;
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(maxidx, m);
}

// ----------------------------------------------------------------------------- step
// step!(env, s, a; track) for one instance per thread.  FROM_SERIES: the exogenous state fields are
// taken from series row idx (they equal env.state there after reset!/step!); otherwise from obs
// (after shems_set_state injected an arbitrary state).
// measured (profiles/r2_step_kernel.md): 128 threads x 10 blocks/SM (48 registers, no spills) is the fastest of the sweep
#ifndef STEP_THREADS
#define STEP_THREADS 128
#endif
#ifndef STEP_MIN_BLOCKS
#define STEP_MIN_BLOCKS 10
#endif
template <bool FROM_SERIES, bool WANT_TRACE, bool FAST>
__global__ void __launch_bounds__(STEP_THREADS, STEP_MIN_BLOCKS)
shems_step_kernel(DevParams P, const float4* __restrict__ series, long long N, float* __restrict__ obs,
                  int32_t* __restrict__ idx_arr, const float* __restrict__ act, int track_neg,
                  float* __restrict__ reward_out, double* __restrict__ reward64_out, float* __restrict__ obs_out, double* __restrict__ trace,
                  long long n0, long long n1) {
  const long long n = n0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n1) return;
  const int idx = idx_arr[n];
  const float a0 = act[n], a1 = act[N + n];
  StepIn s;
  s.Soc_b = obs[0 * N + n];
  s.Soc_ev = obs[1 * N + n];
  float cd_here;
  if (FROM_SERIES) {
    const Row8 r = load_row(series, idx);
    s.c_ev = r.cd; s.d_e = r.d_e; s.g_e = r.g_e; s.p_buy = r.p_buy;
    cd_here = r.cd;
  } else {
    s.c_ev = obs[2 * N + n]; s.d_e = obs[3 * N + n]; s.g_e = obs[4 * N + n]; s.p_buy = obs[5 * N + n];
    cd_here = __ldg(&reinterpret_cast<const float*>(series)[8 * (size_t)(idx - 1) + 1]);  // df[env.idx, :h_countdown] :270
  }
  float B, EV, Bt, EVt;
  if (!track_neg) {  // :346-349
    Bt = a0; EVt = a1;
    shems_action_drl<FAST>(P, s.Soc_b, s.Soc_ev, s.c_ev, s.d_e, s.g_e, Bt, EVt, B, EV);
  } else {           // :350-353
    Bt = 0.0f; EVt = 0.0f; B = a0; EV = a1;
  }
  StepTrace tr;
  const StepOut o = shems_flows<WANT_TRACE, FAST>(P, s, B, EV, EVt, track_neg != 0, &tr);
  // next_state! :264-281
  const Row8 nx = load_row(series, idx + 1);
  const float Soc_ev_new = next_soc_ev(o.Soc_ev, nx, cd_here);
  store_obs(obs, N, n, o.Soc_b, Soc_ev_new, nx);
  idx_arr[n] = idx + 1;  // :456
  if (reward_out) reward_out[n] = (float)o.reward;
  if (reward64_out) reward64_out[n] = o.reward;  // env.reward::Float64 (:171, :467-470)
  if (obs_out) store_obs(obs_out, N, n, o.Soc_b, Soc_ev_new, nx);
  if (WANT_TRACE) store_trace_row(trace + n, N, idx, s, Bt, EVt, o, tr);
}

// action(env, track) / action(env, a) for all instances
template <bool RULE>
__global__ void __launch_bounds__(256)
shems_action_kernel(DevParams P, long long N, const float* __restrict__ obs, const float* __restrict__ target, float* __restrict__ bev,
                    long long n0, long long n1) {
  const long long n = n0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n1) return;
  float B, EV;
  if (RULE) shems_action_rule<false>(P, obs[0 * N + n], obs[1 * N + n], obs[3 * N + n], obs[4 * N + n], B, EV);
  else shems_action_drl<false>(P, obs[0 * N + n], obs[1 * N + n], obs[2 * N + n], obs[3 * N + n], obs[4 * N + n], target[n], target[N + n], B, EV);
  bev[n] = B;
  bev[N + n] = EV;
}

// ----------------------------------------------------------------------------- fused rollout
// T transitions per instance with the state kept in registers (episode!/populate_memory/inference
// loops: DDPG.jl:186-242, memory_plotting_saving.jl:9-29, 62-89).  One thread per instance.
struct RolloutSinks {
  double* ep_return;   // [N]
  double* trace;       // [T][23][N]
  float* obs_traj;     // [T][9][N]
  float* reward_traj;  // [T][N]
  float* ring;         // replay ring (tiled SoA, ring.cuh), capacity cap, first slot `head`
  long long cap, head;
  uint32_t src_entry;  // COMPACT: the ring's series-table entry of this group's series, pre-shifted (ring_tag(entry, 0))
};

// Occupancy matters more than anything else here (measured, profiles/r1_rollout_sweep.md): 128 threads x >= 6 blocks/SM
// caps the kernel at 80 registers -> 24 warps/SM, enough to cover the FP64/XU latencies; at the compiler's
// unconstrained 115 registers (8 warps/SM) the same code runs at half the speed.
#ifndef ROLLOUT_THREADS
#define ROLLOUT_THREADS 128
#endif
#ifndef ROLLOUT_MIN_BLOCKS
#define ROLLOUT_MIN_BLOCKS 6
#endif
// MINB = resident CTAs per SM the register budget is cut for (6: 80 registers, 7: 72, 8: 64).  6 is the fastest per wave; 7 or 8 are
// chosen when they save a mostly empty last wave (e.g. 2^20 instances over 8 GPUs = 1024 CTAs per GPU: 1.15 waves of 148 x 6 CTAs,
// but ONE wave of 148 x 7) — see rollout_min_blocks().
// The rollout policy's action for instance n at step t of a launch, from state s on a row of class CLS: the feasible (B, EV), the
// targets (Bt, EVt) step! records, the action remember() stores (a_raw) and track < 0.  The random policy takes Philox words w0, w1.
struct RolloutAction { float B, EV, Bt, EVt, a_raw0, a_raw1; bool track_neg; };
template <int POLICY, bool FAST, int CLS = ROW_ANY>
__device__ __forceinline__ RolloutAction rollout_action(const DevParams& P, const StepIn& s, uint32_t w0, uint32_t w1,
                                                        const float* __restrict__ tape, int tape_unscaled, long long N, long long n, int t) {
  RolloutAction a;
  a.track_neg = false;
  if (POLICY == SHEMS_POLICY_RULE) {  // DDPG.jl:209-212
    shems_action_rule<FAST>(P, s.Soc_b, s.Soc_ev, s.d_e, s.g_e, a.B, a.EV);
    a.Bt = 0.0f; a.EVt = 0.0f; a.a_raw0 = a.B; a.a_raw1 = a.EV; a.track_neg = true;
    return a;
  }
  if (POLICY == SHEMS_POLICY_RANDOM) {  // memory_plotting_saving.jl:14-19: u = w * 2^-32; a = Float32(2u - 1) (action_from_word, philox.cuh)
    a.a_raw0 = action_from_word(w0);
    a.a_raw1 = action_from_word(w1);
    // scale_action with bounds (0,0)/(1,1) (DDPG.jl:178-184, input.jl:182-183): Float32((Float64(a) + 1.0) * 0.5).
    // a is a multiple of 2^-31, so a + 1.0 and the halving are exact in Float64 and the single final rounding
    // equals the Float32 add followed by the exact halving.
    a.Bt = (a.a_raw0 + 1.0f) * 0.5f;
    a.EVt = (a.a_raw1 + 1.0f) * 0.5f;
  } else {
    a.Bt = tape[((size_t)t * 2 + 0) * N + n];
    a.EVt = tape[((size_t)t * 2 + 1) * N + n];
    a.a_raw0 = a.Bt; a.a_raw1 = a.EVt;
    if (tape_unscaled) {  // the tape holds what `remember` stores (DDPG.jl:229): a in [-1,1]; scale_action with bounds (0,0)/(1,1)
      a.Bt = (float)(((double)a.a_raw0 + 1.0) * 0.5);   // Float32.(lo .+ (a .+ ones(2)) .* 0.5 .* (hi .- lo))  (:178-184)
      a.EVt = (float)(((double)a.a_raw1 + 1.0) * 0.5);
    }
  }
  shems_action_drl<FAST, CLS>(P, s.Soc_b, s.Soc_ev, s.c_ev, s.d_e, s.g_e, a.Bt, a.EVt, a.B, a.EV);
  return a;
}

// COMPACT: the ring sink stores 8 words per transition (Soc_b, Soc_ev, a, r, Soc_b', Soc_ev', series tag; ring.cuh) instead of 23 —
// only when s[2..8] is series row idx, i.e. the env is consistent.
template <int POLICY, bool WANT_TRACE, int MINB, bool FAST, bool COMPACT>
__global__ void __launch_bounds__(ROLLOUT_THREADS, MINB)
shems_rollout_kernel(DevParams P, const float4* __restrict__ series, long long N, float* __restrict__ obs,
                     int32_t* __restrict__ idx_arr, int T, int step0, unsigned long long seed, long long env_id_base,
                     const float* __restrict__ tape, int tape_unscaled, RolloutSinks S, long long n0, long long n1) {
  const long long n = n0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n1) return;
  int idx = idx_arr[n];
  float st[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) st[k] = obs[k * N + n];
  float cd_here = __ldg(&reinterpret_cast<const float*>(series)[8 * (size_t)(idx - 1) + 1]);
  double ret = 0.0;
  long long slot = 0;
  if (S.ring) { slot = S.head + n; if (slot >= S.cap) slot -= S.cap; }  // head < cap, n < N <= cap
  uint32_t rw[4] = {0u, 0u, 0u, 0u};
  for (int t = 0; t < T; ++t) {
    StepIn s;
    s.Soc_b = st[0]; s.Soc_ev = st[1]; s.c_ev = st[2]; s.d_e = st[3]; s.g_e = st[4]; s.p_buy = st[5];
    uint32_t w0 = 0u, w1 = 0u;
    if (POLICY == SHEMS_POLICY_RANDOM) {  // one Philox block per two steps: words 0..1 serve the even step, words 2..3 the odd one
      const unsigned st_abs = (unsigned)(step0 + t);
      if (t == 0 || (st_abs & 1u) == 0u) philox4x32_10(seed, (uint64_t)(env_id_base + n), st_abs >> 1, STREAM_ACTION, rw);
      w0 = (st_abs & 1u) ? rw[2] : rw[0]; w1 = (st_abs & 1u) ? rw[3] : rw[1];
    }
    const RolloutAction a = rollout_action<POLICY, FAST>(P, s, w0, w1, tape, tape_unscaled, N, n, t);
    StepTrace tr;
    const StepOut o = shems_flows<WANT_TRACE, FAST>(P, s, a.B, a.EV, a.EVt, a.track_neg, &tr);
    const Row8 nx = load_row(series, idx + 1);
    const float Soc_ev_new = next_soc_ev(o.Soc_ev, nx, cd_here);
    if (S.ring) {  // remember(s, a, r, s', finished) — memory_plotting_saving.jl:46-47; stores at fixed 128-byte strides
      float* q = S.ring + ring_base(slot);
      if (COMPACT) {  // s[2..8] = series row idx, s'[2..8] = row idx + 1, done = 0: the tag names them
        ring_store_compact(q, st[0], st[1], a.a_raw0, a.a_raw1, (float)o.reward, o.Soc_b, Soc_ev_new, S.src_entry, idx);
      } else {
        // sv copies st: passing st itself takes its address, and the kernel then compiles to a different register allocation
        const float sv[9] = {st[0], st[1], st[2], st[3], st[4], st[5], st[6], st[7], st[8]};
        const float s2v[9] = {o.Soc_b, Soc_ev_new, nx.cd, nx.d_e, nx.g_e, nx.p_buy, nx.h_cos, nx.h_sin, nx.season};
        ring_store_full(q, sv, a.a_raw0, a.a_raw1, (float)o.reward, s2v, 0.0f);  // finished() is always false (shems_LU1.jl:487-502)
      }
      slot += N;
      if (slot >= S.cap) slot -= S.cap;
    }
    if (WANT_TRACE) store_trace_row(S.trace + (size_t)t * SHEMS_TRACE_COLS * N + n, N, idx, s, a.Bt, a.EVt, o, tr);
    st[0] = o.Soc_b; st[1] = Soc_ev_new; st[2] = nx.cd; st[3] = nx.d_e; st[4] = nx.g_e; st[5] = nx.p_buy;
    st[6] = nx.h_cos; st[7] = nx.h_sin; st[8] = nx.season;
    cd_here = nx.cd;
    idx += 1;
    ret += o.reward;  // reward_eps += r (DDPG.jl:223; Float64 accumulation)
    if (S.obs_traj) {
#pragma unroll
      for (int k = 0; k < 9; ++k) S.obs_traj[((size_t)t * 9 + k) * N + n] = st[k];
    }
    if (S.reward_traj) S.reward_traj[(size_t)t * N + n] = (float)o.reward;
  }
#pragma unroll
  for (int k = 0; k < 9; ++k) obs[k * N + n] = st[k];
  idx_arr[n] = idx;
  if (S.ep_return) S.ep_return[n] = ret;
}

// The same rollout, trimmed for the launches that need none of the general kernel's options: FAST constants, a consistent env
// (s[2..8] is series row idx, so only the four row fields the step reads are carried and the final obs write loads the last row
// once), no trace, no obs trajectory, and either no ring or compact records with N and cap multiples of 32 (RingWalk).  One Philox
// block serves two steps: the loop advances two steps per block, starting one step early when step0 is odd, and the round keys come
// precomputed from the host.  Every output bit equals shems_rollout_kernel's.
// Lock step: a warp whose instances all stand at the same row when the launch starts stays in step with itself (every instance
// advances one row per step), so the row class (shems_device.cuh) is uniform across it at every step.  Such a warp (when `lockstep`
// allows it) runs a loop that dispatches each step to the body compiled for the row's class.  That loop advances one step per
// iteration, so each class body is inlined once (about 19 KB of loop); the Philox block is drawn on even steps and its words 2..3
// serve the odd one.  Two steps per iteration with every body inlined twice was measured faster in lock step but slower on the
// two-step loop (profiles/r6_lockstep_rollout.md).  Any other warp runs the two-step loop with the general body only.  Each lane
// takes its own row's class, so the bits never depend on the vote: it only decides the speed.
// When the host knows that every instance of the launch stands on one row (ShemsEnv::uniform_row) and the grid is large enough,
// shems_rollout_pair_kernel below runs this lock-step loop with two instances per thread instead (profiles/r10_pair_rollout.md).
template <int CLS> struct RowTag { static constexpr int value = CLS; };
// f(RowTag<cls>{}): the body of f compiled for the row class cls
template <class F>
__device__ __forceinline__ void with_row_class(int cls, F&& f) {
  switch (cls) {
    case ROW_A_NOEV: f(RowTag<ROW_A_NOEV>{}); break;
    case ROW_B_NOEV: f(RowTag<ROW_B_NOEV>{}); break;
    case ROW_A_EV: f(RowTag<ROW_A_EV>{}); break;
    case ROW_B_EV: f(RowTag<ROW_B_EV>{}); break;
    default: f(RowTag<ROW_ANY>{}); break;
  }
}
// The lock-step loops' random words for step t of I consecutive instances (Philox ids id, id + 1, ...): rw holds I blocks of 4 words,
// and words 0..1 of block i serve instance i.  Block (step0 + t) / 2 is drawn on an even step (and at t = 0); an odd step moves its
// words 2..3 to 0..1.  rw is a flat pointer: taken as an array of I blocks, the trimmed kernel's random-policy builds compile differently.
template <int I>
__device__ __forceinline__ void lockstep_words(const PhiloxKeys& K, uint64_t id, int step0, int t, uint32_t* rw) {
  const unsigned st_abs = (unsigned)(step0 + t);
  if ((st_abs & 1u) == 0u || t == 0) {
#pragma unroll
    for (int i = 0; i < I; ++i) philox4x32_10(K, id + i, st_abs >> 1, STREAM_ACTION, rw + 4 * i);
  }
  if (st_abs & 1u) {
#pragma unroll
    for (int i = 0; i < I; ++i) { rw[4 * i + 0] = rw[4 * i + 2]; rw[4 * i + 1] = rw[4 * i + 3]; }
  }
}
template <int POLICY, int MINB>
__global__ void __launch_bounds__(ROLLOUT_THREADS, MINB)
shems_rollout_lean_kernel(DevParams P, const float4* __restrict__ series, long long N, float* __restrict__ obs,
                          int32_t* __restrict__ idx_arr, int T, int step0, PhiloxKeys K, long long env_id_base,
                          const float* __restrict__ tape, int tape_unscaled, RolloutSinks S, long long n0, long long n1, int lockstep) {
  const long long n = n0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n1) return;
  int idx = idx_arr[n];
  float Soc_b = obs[0 * N + n], Soc_ev = obs[1 * N + n];
  float c_ev, d_e, g_e, p_buy;
  { const Row8 r = load_row(series, idx); c_ev = r.cd; d_e = r.d_e; g_e = r.g_e; p_buy = r.p_buy; }
  double ret = 0.0;
  RingWalk ring{};
  if (S.ring) { long long slot = S.head + n; if (slot >= S.cap) slot -= S.cap; ring = ring_walk(S.ring, slot, N, S.cap); }
  const uint64_t id = (uint64_t)(env_id_base + n);
  auto step = [&](auto cls, int t, uint32_t w0, uint32_t w1) {
    constexpr int CLS = decltype(cls)::value;
    StepIn s;
    s.Soc_b = Soc_b; s.Soc_ev = Soc_ev; s.c_ev = c_ev; s.d_e = d_e; s.g_e = g_e; s.p_buy = p_buy;
    const RolloutAction a = rollout_action<POLICY, true, CLS>(P, s, w0, w1, tape, tape_unscaled, N, n, t);
    StepTrace tr;
    const StepOut o = shems_flows<false, true, CLS>(P, s, a.B, a.EV, a.EVt, a.track_neg, &tr);
    const Row8 nx = load_row(series, idx + 1);
    const float Soc_ev_new = next_soc_ev<CLS>(o.Soc_ev, nx, c_ev);
    if (S.ring) {
      ring_store_compact(ring.q, Soc_b, Soc_ev, a.a_raw0, a.a_raw1, (float)o.reward, o.Soc_b, Soc_ev_new, S.src_entry, idx);
      ring_walk_next(ring);
    }
    if (S.reward_traj) S.reward_traj[(size_t)t * N + n] = (float)o.reward;
    Soc_b = o.Soc_b; Soc_ev = Soc_ev_new; c_ev = nx.cd; d_e = nx.d_e; g_e = nx.g_e; p_buy = nx.p_buy;
    idx += 1;
    ret += o.reward;
  };
  // the lanes that returned above are not in the mask (N need not be a multiple of 32 without a ring)
  const unsigned mask = __activemask();
  if (lockstep && __all_sync(mask, idx == __shfl_sync(mask, idx, __ffs(mask) - 1))) {
    uint32_t rw[4] = {0u, 0u, 0u, 0u};
    for (int t = 0; t < T; ++t) {
      if (POLICY == SHEMS_POLICY_RANDOM) lockstep_words<1>(K, id, step0, t, rw);
      with_row_class(row_class(P, c_ev, d_e, g_e), [&](auto cls) { step(cls, t, rw[0], rw[1]); });
    }
  } else {
    // t is the step that uses words 0..1 of the block; with an odd step0 the first block's words 0..1 belong to step -1
    for (int t = POLICY == SHEMS_POLICY_RANDOM ? -(step0 & 1) : 0; t < T; t += 2) {
      uint32_t rw[4] = {0u, 0u, 0u, 0u};
      if (POLICY == SHEMS_POLICY_RANDOM) philox4x32_10(K, id, (unsigned)(step0 + t) >> 1, STREAM_ACTION, rw);
      if (t >= 0) step(RowTag<ROW_ANY>{}, t, rw[0], rw[1]);
      if (t + 1 < T) step(RowTag<ROW_ANY>{}, t + 1, rw[2], rw[3]);
    }
  }
  store_obs(obs, N, n, Soc_b, Soc_ev, load_row(series, idx));
  idx_arr[n] = idx;
  if (S.ep_return) S.ep_return[n] = ret;
}

// The lock-step loop of shems_rollout_lean_kernel with two instances per thread, for launches in which every instance stands on the
// same row (ShemsEnv::uniform_row, so no vote and no other loop).  Thread k carries instances n0 + 2k and n0 + 2k + 1: the row class
// and its dispatch, the next row's load, the terms of the step that depend on the row only (both instances' bodies sit in one class
// body, so the compiler computes those once), the loop control and the ring walk are paid once for two instances.  Each instance keeps
// its own Soc_b, Soc_ev, return and Philox stream (id = env_id_base + its index).  With a ring, head + n0 is even, so the two records
// sit in adjacent slots of one tile and each field of both is one 8-byte store.  Every output bit equals shems_rollout_lean_kernel's.
template <int POLICY, int MINB>
__global__ void __launch_bounds__(ROLLOUT_THREADS, MINB)
shems_rollout_pair_kernel(DevParams P, const float4* __restrict__ series, long long N, float* __restrict__ obs,
                          int32_t* __restrict__ idx_arr, int T, int step0, PhiloxKeys K, long long env_id_base,
                          const float* __restrict__ tape, int tape_unscaled, RolloutSinks S, long long n0, long long n1) {
  const long long n = n0 + 2 * ((long long)blockIdx.x * blockDim.x + threadIdx.x);
  if (n >= n1) return;  // n1 - n0 is even
  int idx = idx_arr[n];
  float Soc_b[2] = {obs[n], obs[n + 1]}, Soc_ev[2] = {obs[N + n], obs[N + n + 1]};
  float c_ev, d_e, g_e, p_buy;
  { const Row8 r = load_row(series, idx); c_ev = r.cd; d_e = r.d_e; g_e = r.g_e; p_buy = r.p_buy; }
  double ret[2] = {0.0, 0.0};
  RingWalk ring{};
  if (S.ring) { long long slot = S.head + n; if (slot >= S.cap) slot -= S.cap; ring = ring_walk(S.ring, slot, N, S.cap); }
  const uint64_t id = (uint64_t)(env_id_base + n);
  auto step = [&](auto cls, int t, const uint32_t (&rw)[2][4]) {
    constexpr int CLS = decltype(cls)::value;
    const Row8 nx = load_row(series, idx + 1);
    float a_raw0[2], a_raw1[2], r32[2], Soc_b2[2], Soc_ev2[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      StepIn s;
      s.Soc_b = Soc_b[i]; s.Soc_ev = Soc_ev[i]; s.c_ev = c_ev; s.d_e = d_e; s.g_e = g_e; s.p_buy = p_buy;
      const RolloutAction a = rollout_action<POLICY, true, CLS>(P, s, rw[i][0], rw[i][1], tape, tape_unscaled, N, n + i, t);
      a_raw0[i] = a.a_raw0; a_raw1[i] = a.a_raw1;
      StepTrace tr;
      const StepOut o = shems_flows<false, true, CLS>(P, s, a.B, a.EV, a.EVt, a.track_neg, &tr);
      Soc_ev2[i] = next_soc_ev<CLS>(o.Soc_ev, nx, c_ev);
      Soc_b2[i] = o.Soc_b;
      r32[i] = (float)o.reward;
      ret[i] += o.reward;
    }
    if (S.ring) {
      ring_store_compact_pair(ring.q, Soc_b, Soc_ev, a_raw0, a_raw1, r32, Soc_b2, Soc_ev2, S.src_entry, idx);
      ring_walk_next(ring);
    }
    if (S.reward_traj) { S.reward_traj[(size_t)t * N + n] = r32[0]; S.reward_traj[(size_t)t * N + n + 1] = r32[1]; }
#pragma unroll
    for (int i = 0; i < 2; ++i) { Soc_b[i] = Soc_b2[i]; Soc_ev[i] = Soc_ev2[i]; }
    c_ev = nx.cd; d_e = nx.d_e; g_e = nx.g_e; p_buy = nx.p_buy;
    idx += 1;
  };
  uint32_t rw[2][4] = {};
  for (int t = 0; t < T; ++t) {
    if (POLICY == SHEMS_POLICY_RANDOM) lockstep_words<2>(K, id, step0, t, &rw[0][0]);
    with_row_class(row_class(P, c_ev, d_e, g_e), [&](auto cls) { step(cls, t, rw); });
  }
  const Row8 r = load_row(series, idx);
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    store_obs(obs, N, n + i, Soc_b[i], Soc_ev[i], r);
    idx_arr[n + i] = idx;
    if (S.ep_return) S.ep_return[n + i] = ret[i];
  }
}

// ----------------------------------------------------------------------------- C ABI
static inline unsigned grid_for(long long n, int block) { return (unsigned)((n + block - 1) / block); }

// The integer value of environment variable `name`, `dflt` when it is unset.  The A/B switches of the rollout (SHEMS_RING_COMPACT,
// SHEMS_ROLLOUT_LEAN, SHEMS_ROLLOUT_LOCKSTEP, SHEMS_ROLLOUT_PAIR; see shems_rollout) are read at every rollout, so that bit-equality
// tests and same-process timings can flip them between calls.
static int env_int(const char* name, int dflt) {
  const char* ev = getenv(name);
  return ev ? atoi(ev) : dflt;
}

// Resident CTAs per SM for a rollout over n instances.  A wave of 148 x b CTAs takes about the same time for b = 6, 7, 8 per CTA slot
// (measured: 6 is 1-3 % faster per instance, profiles/r1_rollout_sweep.md), but a sparsely filled LAST wave runs its few warps at a
// fraction of the issue rate: cost model = full waves + the last wave's fill, floored at 0.45 (a lone warp per scheduler is latency
// bound), times the per-instance penalty of the tighter register budget.  That model was measured on the store-bound kernel that
// writes full ring records.  With compact records the kernel is issue bound and its MINB = 6 build needs only 66 registers (7 CTAs
// per SM anyway); it was the fastest of 6 / 7 / 8 at 2^20 and at 2^17 instances (profiles/r3_ring_compact.md), so compact launches
// take 6.  The trimmed kernel (shems_rollout_lean_kernel) needs 78 registers for the random policy at MINB 6, which leaves 6 CTAs per
// SM; at MINB 7 it fits 72 without spilling and keeps 7, so its compact launches take 7 (profiles/r5_lean_rollout.md).
// SHEMS_ROLLOUT_MIN_BLOCKS=6|7|8 overrides.
static int sm_count(int device) {
  static int sms[64];
  if (device >= 0 && device < 64 && sms[device] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || v <= 0) { cudaGetLastError(); v = 148; }
    sms[device] = v;
  }
  return (device >= 0 && device < 64) ? sms[device] : 148;
}
static int rollout_min_blocks(int device, long long n, bool compact, bool lean) {
  static const int forced = env_int("SHEMS_ROLLOUT_MIN_BLOCKS", 0);
  if (forced == 6 || forced == 7 || forced == 8) return forced;
  if (compact) return lean ? 7 : 6;
  const int nsm = sm_count(device);
  const double ctas = (double)((n + ROLLOUT_THREADS - 1) / ROLLOUT_THREADS);
  int best = ROLLOUT_MIN_BLOCKS; double best_cost = 1e300;
  for (int b = 6; b <= 8; ++b) {
    const double waves = ctas / ((double)nsm * b);
    const double full = floor(waves), frac = waves - full;
    const double last = frac > 0.0 ? (frac < 0.45 ? 0.45 : frac) : 0.0;
    const double penalty = b == 6 ? 1.0 : (b == 7 ? 1.015 : 1.03);
    const double cost = (full + last) * b * penalty;   // time ~ waves x (instances per wave ~ b)
    if (cost < best_cost - 1e-9) { best_cost = cost; best = b; }
  }
  return best;
}

// The pair kernel (shems_rollout_pair_kernel) applies to a launch the trimmed kernel would take in lock step whose instances all stand
// on one row, with an even count and, with a ring, an even first slot.  It is taken there when its grid of half as many threads fills
// at least ROLLOUT_PAIR_MIN_WAVES waves of ROLLOUT_PAIR_MIN_BLOCKS CTAs per SM: below that, the trimmed kernel's grid of twice the
// warps hides the step's latencies better (profiles/r10_pair_rollout.md).  SHEMS_ROLLOUT_PAIR=0 forces the trimmed kernel and
// SHEMS_ROLLOUT_PAIR=2 takes the pair kernel wherever it applies, whatever the grid (read at every rollout: the A/B switch, and
// small launches for bit-equality tests).
#ifndef ROLLOUT_PAIR_MIN_BLOCKS
#define ROLLOUT_PAIR_MIN_BLOCKS 4
#endif
#ifndef ROLLOUT_PAIR_MIN_WAVES
#define ROLLOUT_PAIR_MIN_WAVES 1
#endif
static bool rollout_pair_fills(int device, long long n, int mode) {
  if (mode == 2) return true;
  const long long ctas = (n / 2 + ROLLOUT_THREADS - 1) / ROLLOUT_THREADS;
  return ctas >= (long long)ROLLOUT_PAIR_MIN_WAVES * sm_count(device) * ROLLOUT_PAIR_MIN_BLOCKS;
}
// pair-kernel launches this process has made (tests use it to tell which kernel ran)
static long long g_pair_launches = 0;
extern "C" int64_t shems_rollout_pair_launches(void) { return __atomic_load_n(&g_pair_launches, __ATOMIC_RELAXED); }

// Shems(maxsteps, path) for G groups of instances (group g: group_sizes[g] consecutive instances with params[g] and, when
// series_per_group, its own series): several chargers in one handle.  Every kernel is launched once per group on its slice.
extern "C" int32_t shems_create_groups(const ShemsParams* params, int32_t n_groups, const int64_t* group_sizes, const float* series_host,
                                       int32_t series_per_group, int32_t nrows, int32_t maxsteps, int32_t device, ShemsEnv** out) {
  REQUIRE(params && series_host && out && group_sizes, SHEMS_ERR_INVALID, "shems_create: NULL argument");
  REQUIRE(n_groups >= 1 && n_groups <= SHEMS_MAX_GROUPS, SHEMS_ERR_INVALID, "shems_create: n_groups=%d (1..%d)", n_groups, SHEMS_MAX_GROUPS);
  int64_t n_envs = 0;
  for (int g = 0; g < n_groups; ++g) {
    REQUIRE(group_sizes[g] >= 1, SHEMS_ERR_INVALID, "shems_create: group_sizes[%d]=%lld", g, (long long)group_sizes[g]);
    n_envs += group_sizes[g];
  }
  REQUIRE(nrows >= 2 && maxsteps >= 1, SHEMS_ERR_INVALID, "shems_create: nrows=%d maxsteps=%d", nrows, maxsteps);
  REQUIRE(nrows - maxsteps >= 1, SHEMS_ERR_INVALID,
          "shems_create: nrows - maxsteps = %d < 1: rand(1:(nrow-maxsteps)) would be empty (shems_LU1.jl:225)", nrows - maxsteps);
  REQUIRE(shems_device_count() > 0, SHEMS_ERR_CUDA, "shems_create: no CUDA device (this library has no CPU fallback)");
  GUARD(device);
  ShemsEnv* e = new (std::nothrow) ShemsEnv();
  REQUIRE(e, SHEMS_ERR_INVALID, "shems_create: out of host memory");
  memset(e, 0, sizeof(*e));
  e->device = device; e->stream = 0; e->params = params[0]; e->dp = make_dev_params(params[0]);
  e->nrows = nrows; e->maxsteps = maxsteps; e->n = n_envs; e->max_idx = 1; e->consistent = true;
  e->n_groups = n_groups;
  static unsigned long long next_serial = 0;
  e->serial = __atomic_add_fetch(&next_serial, 1, __ATOMIC_RELAXED);
  const int n_series = series_per_group ? n_groups : 1;
  // interleave the 8 columns into 32-byte rows
  std::vector<float> rows((size_t)n_series * nrows * 8);
  for (int g = 0; g < n_series; ++g)
    for (int r = 0; r < nrows; ++r)
      for (int c = 0; c < 8; ++c) rows[((size_t)g * nrows + r) * 8 + c] = series_host[((size_t)g * 8 + c) * nrows + r];
  cudaError_t st = cudaSuccess;
  if ((st = cudaMalloc(&e->series, sizeof(float) * rows.size())) != cudaSuccess ||
      (st = cudaMalloc(&e->obs, sizeof(float) * 9 * (size_t)n_envs)) != cudaSuccess ||
      (st = cudaMalloc(&e->idx, sizeof(int32_t) * (size_t)n_envs)) != cudaSuccess ||
      (st = cudaMalloc(&e->d_maxidx, sizeof(int32_t))) != cudaSuccess ||
      (st = cudaMemcpy(e->series, rows.data(), sizeof(float) * rows.size(), cudaMemcpyHostToDevice)) != cudaSuccess ||
      (st = cudaMemset(e->obs, 0, sizeof(float) * 9 * (size_t)n_envs)) != cudaSuccess ||
      (st = cudaMemset(e->idx, 0, sizeof(int32_t) * (size_t)n_envs)) != cudaSuccess) {
    shems_set_error("shems_create: %s", cudaGetErrorString(st));
    shems_destroy(e);
    return SHEMS_ERR_CUDA;
  }
  if ((st = cudaMallocHost((void**)&e->h_maxidx, sizeof(int32_t))) != cudaSuccess ||
      (st = cudaEventCreateWithFlags(&e->ev_maxidx, cudaEventDisableTiming)) != cudaSuccess) {
    shems_set_error("shems_create: %s", cudaGetErrorString(st));
    shems_destroy(e);
    return SHEMS_ERR_CUDA;
  }
  for (int g = 0; g < n_groups; ++g) {
    e->gdp[g] = make_dev_params(params[g]);
    e->gseries[g] = e->series + (series_per_group ? (size_t)g * nrows * 2 : 0);
    e->gstart[g + 1] = e->gstart[g] + group_sizes[g];
  }
  *out = e;
  return SHEMS_OK;
}

extern "C" int32_t shems_create(const ShemsParams* params, const float* series_host, int32_t nrows, int32_t maxsteps,
                                int64_t n_envs, int32_t device, ShemsEnv** out) {
  REQUIRE(n_envs >= 1, SHEMS_ERR_INVALID, "shems_create: n_envs=%lld", (long long)n_envs);
  return shems_create_groups(params, 1, &n_envs, series_host, 0, nrows, maxsteps, device, out);
}

extern "C" int32_t shems_destroy(ShemsEnv* e) {
  if (!e) return SHEMS_OK;
  GUARD(e->device);
  cudaFree(e->series); cudaFree(e->obs); cudaFree(e->idx); cudaFree(e->d_maxidx); cudaFree(e->scratch_i); cudaFree(e->scratch_f);
  if (e->h_maxidx) cudaFreeHost(e->h_maxidx);
  if (e->ev_maxidx) cudaEventDestroy(e->ev_maxidx);
  delete e;
  return SHEMS_OK;
}

extern "C" int32_t shems_set_stream(ShemsEnv* e, void* s) {
  REQUIRE(e, SHEMS_ERR_INVALID, "shems_set_stream: NULL handle");
  e->stream = (cudaStream_t)s;
  return SHEMS_OK;
}
extern "C" int32_t shems_sync(ShemsEnv* e) {
  REQUIRE(e, SHEMS_ERR_INVALID, "shems_sync: NULL handle");
  GUARD(e->device);
  CUDA_TRY(cudaStreamSynchronize(e->stream));
  return SHEMS_OK;
}
extern "C" int64_t shems_num_envs(const ShemsEnv* e) { return e ? e->n : 0; }
extern "C" int32_t shems_num_rows(const ShemsEnv* e) { return e ? e->nrows : 0; }
extern "C" int32_t shems_get_step(const ShemsEnv* e, int32_t* step) {
  REQUIRE(e && step, SHEMS_ERR_INVALID, "shems_get_step: NULL argument");
  *step = e->step;
  return SHEMS_OK;
}
extern "C" int32_t shems_finished(const ShemsEnv* e, int32_t* out) {
  REQUIRE(e && out, SHEMS_ERR_INVALID, "shems_finished: NULL argument");
  *out = 0;  // shems_LU1.jl:487-502 returns false on both paths
  return SHEMS_OK;
}

// may the instances advance `need` more rows?  0 = yes; otherwise the row the furthest instance would read (for the message)
int32_t ensure_rows(ShemsEnv* e, int64_t need) {
  if ((int64_t)e->max_idx + need <= e->nrows) return 0;
  if (e->max_pending) {  // the upper bound does not settle it: wait for the exact maximum of the last reset
    cudaEventSynchronize(e->ev_maxidx);
    e->max_idx = *e->h_maxidx + e->step;
    e->max_pending = false;
    if ((int64_t)e->max_idx + need <= e->nrows) return 0;
  }
  return e->max_idx;
}

extern "C" int32_t shems_reset(ShemsEnv* e, int32_t mode, const int32_t* idx0_host, const float* socb0_host, uint64_t seed,
                               int64_t env_id_base) {
  REQUIRE(e, SHEMS_ERR_INVALID, "shems_reset: NULL handle");
  REQUIRE(mode >= 0 && mode <= 2, SHEMS_ERR_INVALID, "shems_reset: unknown mode %d", mode);
  GUARD(e->device);
  const int hi = e->nrows - e->maxsteps;
  if (mode == SHEMS_RESET_HOST_DRAWS) {
    REQUIRE(idx0_host && socb0_host, SHEMS_ERR_INVALID, "shems_reset: HOST_DRAWS needs idx0_host and socb0_host");
    for (int64_t i = 0; i < e->n; ++i)
      REQUIRE(idx0_host[i] >= 1 && idx0_host[i] <= hi, SHEMS_ERR_INVALID, "shems_reset: idx0[%lld]=%d outside 1..%d", (long long)i,
              idx0_host[i], hi);
    if (!e->scratch_i) {
      CUDA_TRY(cudaMalloc(&e->scratch_i, sizeof(int32_t) * (size_t)e->n));
      CUDA_TRY(cudaMalloc(&e->scratch_f, sizeof(float) * (size_t)e->n));
    }
    CUDA_TRY(cudaMemcpyAsync(e->scratch_i, idx0_host, sizeof(int32_t) * (size_t)e->n, cudaMemcpyHostToDevice, e->stream));
    CUDA_TRY(cudaMemcpyAsync(e->scratch_f, socb0_host, sizeof(float) * (size_t)e->n, cudaMemcpyHostToDevice, e->stream));
  }
  CUDA_TRY(cudaMemsetAsync(e->d_maxidx, 0, sizeof(int32_t), e->stream));
  for (int g = 0; g < e->n_groups; ++g) {
    const long long n0 = e->gstart[g], n1 = e->gstart[g + 1];
    COUNT_LAUNCH();
    shems_reset_kernel<<<grid_for(n1 - n0, 256), 256, 0, e->stream>>>(e->gdp[g], e->gseries[g], e->nrows, e->maxsteps, e->n, mode, e->scratch_i,
                                                                     e->scratch_f, seed, env_id_base, e->obs, e->idx, e->d_maxidx, n0, n1);
  }
  CUDA_TRY(cudaGetLastError());
  // Bounds pre-check of the following steps (Julia's BoundsError at :266-268) without stalling the host: every start row is
  // <= nrows - maxsteps, which settles every episode of <= maxsteps steps; the exact maximum travels to a pinned word
  // asynchronously and is only waited for when that bound is not enough (ensure_rows).
  if (mode == SHEMS_RESET_DETERMINISTIC) { e->max_idx = 1; e->max_pending = false; }
  else {
    CUDA_TRY(cudaMemcpyAsync(e->h_maxidx, e->d_maxidx, sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
    CUDA_TRY(cudaEventRecord(e->ev_maxidx, e->stream));
    e->max_idx = hi; e->max_pending = true;
  }
  e->step = 0;          // :210
  e->was_reset = true;
  e->consistent = true;
  // one row for every instance: rng = -1, a single admissible start row, or host draws that all name the same row (the window shift
  // of :227-246 depends on the start row only)
  e->uniform_row = mode == SHEMS_RESET_DETERMINISTIC || hi == 1;
  if (mode == SHEMS_RESET_HOST_DRAWS) {
    e->uniform_row = true;
    for (int64_t i = 1; i < e->n && e->uniform_row; ++i) e->uniform_row = idx0_host[i] == idx0_host[0];
  }
  return SHEMS_OK;
}

extern "C" int32_t shems_step(ShemsEnv* e, const float* act_dev, int32_t track, float* reward_dev, double* reward64_dev, float* obs_dev,
                              double* trace_dev) {
  REQUIRE(e && act_dev, SHEMS_ERR_INVALID, "shems_step: NULL argument");
  REQUIRE(e->was_reset, SHEMS_ERR_STATE, "shems_step: reset! (or shems_set_state) must come first");
  if (ensure_rows(e, 1)) {
    shems_set_error("BoundsError: attempt to access %d-row series at row %d (next_state!, shems_LU1.jl:266-268)", e->nrows, e->max_idx + 1);
    return SHEMS_ERR_BOUNDS;
  }
  GUARD(e->device);
  const int tn = track < 0 ? 1 : 0;
#define LAUNCH_STEP(FS, TR)                                                                                                             \
  COUNT_LAUNCH();                                                                                                                       \
  if (!TR && e->gdp[g].fast_all)                                                                                                        \
    shems_step_kernel<FS, false, true><<<grid_for(n1 - n0, STEP_THREADS), STEP_THREADS, 0, e->stream>>>(                                   \
        e->gdp[g], e->gseries[g], e->n, e->obs, e->idx, act_dev, tn, reward_dev, reward64_dev, obs_dev, trace_dev, n0, n1);              \
  else                                                                                                                                  \
    shems_step_kernel<FS, TR, false><<<grid_for(n1 - n0, STEP_THREADS), STEP_THREADS, 0, e->stream>>>(                                     \
        e->gdp[g], e->gseries[g], e->n, e->obs, e->idx, act_dev, tn, reward_dev, reward64_dev, obs_dev, trace_dev, n0, n1)
  for (int g = 0; g < e->n_groups; ++g) {
    const long long n0 = e->gstart[g], n1 = e->gstart[g + 1];
    if (e->consistent) { if (trace_dev) { LAUNCH_STEP(true, true); } else { LAUNCH_STEP(true, false); } }
    else { if (trace_dev) { LAUNCH_STEP(false, true); } else { LAUNCH_STEP(false, false); } }
  }
#undef LAUNCH_STEP
  CUDA_TRY(cudaGetLastError());
  e->max_idx += 1;
  e->step += 1;  // :455
  e->consistent = true;
  return SHEMS_OK;
}

extern "C" int32_t shems_action_rule(ShemsEnv* e, float* bev_dev) {
  REQUIRE(e && bev_dev, SHEMS_ERR_INVALID, "shems_action_rule: NULL argument");
  GUARD(e->device);
  for (int g = 0; g < e->n_groups; ++g, COUNT_LAUNCH())
    shems_action_kernel<true><<<grid_for(e->gstart[g + 1] - e->gstart[g], 256), 256, 0, e->stream>>>(e->gdp[g], e->n, e->obs, nullptr, bev_dev,
                                                                                                    e->gstart[g], e->gstart[g + 1]);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}
extern "C" int32_t shems_action_drl(ShemsEnv* e, const float* target_dev, float* bev_dev) {
  REQUIRE(e && target_dev && bev_dev, SHEMS_ERR_INVALID, "shems_action_drl: NULL argument");
  GUARD(e->device);
  for (int g = 0; g < e->n_groups; ++g, COUNT_LAUNCH())
    shems_action_kernel<false><<<grid_for(e->gstart[g + 1] - e->gstart[g], 256), 256, 0, e->stream>>>(e->gdp[g], e->n, e->obs, target_dev, bev_dev,
                                                                                                     e->gstart[g], e->gstart[g + 1]);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}

extern "C" int32_t shems_state_ptr(ShemsEnv* e, float** obs_dev, int32_t** idx_dev) {
  REQUIRE(e, SHEMS_ERR_INVALID, "shems_state_ptr: NULL handle");
  if (obs_dev) *obs_dev = e->obs;
  if (idx_dev) *idx_dev = e->idx;
  return SHEMS_OK;
}
extern "C" int32_t shems_get_state(ShemsEnv* e, float* obs_host, int32_t* idx_host) {
  REQUIRE(e && obs_host, SHEMS_ERR_INVALID, "shems_get_state: NULL argument");
  GUARD(e->device);
  CUDA_TRY(cudaMemcpyAsync(obs_host, e->obs, sizeof(float) * 9 * (size_t)e->n, cudaMemcpyDeviceToHost, e->stream));
  if (idx_host) CUDA_TRY(cudaMemcpyAsync(idx_host, e->idx, sizeof(int32_t) * (size_t)e->n, cudaMemcpyDeviceToHost, e->stream));
  CUDA_TRY(cudaStreamSynchronize(e->stream));
  return SHEMS_OK;
}
extern "C" int32_t shems_set_state(ShemsEnv* e, const float* obs_host, const int32_t* idx_host) {
  REQUIRE(e && obs_host && idx_host, SHEMS_ERR_INVALID, "shems_set_state: NULL argument");
  GUARD(e->device);
  int32_t mx = 1;
  for (int64_t i = 0; i < e->n; ++i) {
    REQUIRE(idx_host[i] >= 1 && idx_host[i] <= e->nrows, SHEMS_ERR_INVALID, "shems_set_state: idx[%lld]=%d outside 1..%d", (long long)i,
            idx_host[i], e->nrows);
    mx = idx_host[i] > mx ? idx_host[i] : mx;
  }
  CUDA_TRY(cudaMemcpyAsync(e->obs, obs_host, sizeof(float) * 9 * (size_t)e->n, cudaMemcpyHostToDevice, e->stream));
  CUDA_TRY(cudaMemcpyAsync(e->idx, idx_host, sizeof(int32_t) * (size_t)e->n, cudaMemcpyHostToDevice, e->stream));
  CUDA_TRY(cudaStreamSynchronize(e->stream));
  e->max_idx = mx; e->max_pending = false;
  e->was_reset = true;
  e->consistent = false;
  e->uniform_row = true;
  for (int64_t i = 1; i < e->n && e->uniform_row; ++i) e->uniform_row = idx_host[i] == idx_host[0];
  return SHEMS_OK;
}

// shems_rollout_kernel<POL, TR, MB, FAST, COMPACT> for the run-time COMPACT and, without a trace, the run-time MINB mb
using RolloutKernel = void (*)(DevParams, const float4*, long long, float*, int32_t*, int, int, unsigned long long, long long, const float*, int,
                               RolloutSinks, long long, long long);
template <int POL, bool TR, int MB, bool FAST>
static RolloutKernel general_rollout_kernel(bool compact) {
  return compact ? shems_rollout_kernel<POL, TR, MB, FAST, true> : shems_rollout_kernel<POL, TR, MB, FAST, false>;
}
template <int POL, bool FAST>
static RolloutKernel general_rollout_kernel(int mb, bool compact) {
  return mb == 7   ? general_rollout_kernel<POL, false, 7, FAST>(compact)
         : mb == 8 ? general_rollout_kernel<POL, false, 8, FAST>(compact)
                   : general_rollout_kernel<POL, false, ROLLOUT_MIN_BLOCKS, FAST>(compact);
}

// shems_rollout's launch on group g for policy POL: the pair kernel, the trimmed kernel at MINB mb, or the general kernel (a trace
// takes its Float64-constant build at ROLLOUT_MIN_BLOCKS; otherwise MINB mb and FAST when the group's constants allow it)
template <int POL>
static void launch_rollout(const ShemsEnv* e, const ShemsRolloutArgs* a, const RolloutSinks& S, const PhiloxKeys& keys, int lockstep, int g,
                           bool pair, bool lean, bool compact, int mb) {
  const long long n0 = e->gstart[g], n1 = e->gstart[g + 1];
  if (pair) {
    shems_rollout_pair_kernel<POL, ROLLOUT_PAIR_MIN_BLOCKS><<<grid_for((n1 - n0) / 2, ROLLOUT_THREADS), ROLLOUT_THREADS, 0, e->stream>>>(
        e->gdp[g], e->gseries[g], e->n, e->obs, e->idx, a->n_steps, e->step, keys, a->env_id_base, a->tape_dev, a->tape_unscaled, S, n0, n1);
  } else if (lean) {
    const auto k = mb == 7 ? shems_rollout_lean_kernel<POL, 7> : mb == 8 ? shems_rollout_lean_kernel<POL, 8> : shems_rollout_lean_kernel<POL, ROLLOUT_MIN_BLOCKS>;
    k<<<grid_for(n1 - n0, ROLLOUT_THREADS), ROLLOUT_THREADS, 0, e->stream>>>(e->gdp[g], e->gseries[g], e->n, e->obs, e->idx, a->n_steps, e->step,
                                                                           keys, a->env_id_base, a->tape_dev, a->tape_unscaled, S, n0, n1, lockstep);
  } else {
    const RolloutKernel k = a->trace_dev           ? general_rollout_kernel<POL, true, ROLLOUT_MIN_BLOCKS, false>(compact)
                            : e->gdp[g].fast_all ? general_rollout_kernel<POL, true>(mb, compact)
                                                 : general_rollout_kernel<POL, false>(mb, compact);
    k<<<grid_for(n1 - n0, ROLLOUT_THREADS), ROLLOUT_THREADS, 0, e->stream>>>(e->gdp[g], e->gseries[g], e->n, e->obs, e->idx, a->n_steps, e->step,
                                                                           a->seed, a->env_id_base, a->tape_dev, a->tape_unscaled, S, n0, n1);
  }
}

extern "C" int32_t shems_rollout(ShemsEnv* e, const ShemsRolloutArgs* a) {
  REQUIRE(e && a, SHEMS_ERR_INVALID, "shems_rollout: NULL argument");
  REQUIRE(e->was_reset, SHEMS_ERR_STATE, "shems_rollout: reset! must come first");
  REQUIRE(a->n_steps >= 1, SHEMS_ERR_INVALID, "shems_rollout: n_steps=%d", a->n_steps);
  REQUIRE(a->policy >= 0 && a->policy <= 2, SHEMS_ERR_INVALID, "shems_rollout: unknown policy %d", a->policy);
  REQUIRE(a->policy != SHEMS_POLICY_TAPE || a->tape_dev, SHEMS_ERR_INVALID, "shems_rollout: POLICY_TAPE needs tape_dev");
  // remember() stores the UNSCALED action (DDPG.jl:229): a tape of scaled targets must not feed a training memory
  REQUIRE(!(a->policy == SHEMS_POLICY_TAPE && a->replay && !a->tape_unscaled), SHEMS_ERR_INVALID,
          "shems_rollout: POLICY_TAPE with a replay sink needs tape_unscaled = 1 (actions in [-1,1], as remember() stores them)");
  if (ensure_rows(e, a->n_steps)) {
    shems_set_error("BoundsError: rollout of %d steps from row %d leaves the %d-row series (next_state!, shems_LU1.jl:266-268)", a->n_steps,
                    e->max_idx, e->nrows);
    return SHEMS_ERR_BOUNDS;
  }
  GUARD(e->device);
  RolloutSinks S;
  memset(&S, 0, sizeof(S));
  S.ep_return = a->ep_return_dev; S.trace = a->trace_dev; S.obs_traj = a->obs_traj_dev; S.reward_traj = a->reward_traj_dev;
  S.cap = 1;
  const int64_t total = (int64_t)a->n_steps * e->n;
  if (a->replay) {
    ShemsReplay* rp = a->replay;
    REQUIRE(rp->device == e->device, SHEMS_ERR_INVALID, "shems_rollout: replay lives on device %d, env on %d", rp->device, e->device);
    // a slot must only ever be written by one thread inside a launch: either no wrap onto itself, or
    // the wrap lands on the same instance (capacity multiple of N)
    REQUIRE(total <= rp->capacity || rp->capacity % e->n == 0, SHEMS_ERR_INVALID,
            "shems_rollout: replay capacity %lld must hold n_steps*n_envs=%lld or be a multiple of n_envs=%lld", (long long)rp->capacity,
            (long long)total, (long long)e->n);
    REQUIRE(e->n <= rp->capacity, SHEMS_ERR_INVALID, "shems_rollout: replay capacity %lld < n_envs %lld", (long long)rp->capacity, (long long)e->n);
    S.ring = rp->ring; S.cap = rp->capacity; S.head = rp->head;
  }
  // SHEMS_ROLLOUT_LEAN=0 forces the general kernel where the trimmed one would apply
  const bool may_lean = !a->trace_dev && !a->obs_traj_dev && e->consistent && env_int("SHEMS_ROLLOUT_LEAN", 1) != 0;
  const PhiloxKeys keys = philox_keys(a->seed);
  // SHEMS_ROLLOUT_LOCKSTEP=0 keeps every warp of the trimmed kernel on its two-step loop, and so never takes the pair kernel
  const int lockstep = env_int("SHEMS_ROLLOUT_LOCKSTEP", 1) != 0 ? 1 : 0;
  const int pair_mode = lockstep ? env_int("SHEMS_ROLLOUT_PAIR", 1) : 0;
  // compact records need s[2..8] == series row idx (consistent), a row that fits the tag and a series-table entry in the ring;
  // SHEMS_RING_COMPACT=0 forces full ones
  const bool may_compact = a->replay && e->consistent && e->nrows <= RING_TAG_MAX_ROW && env_int("SHEMS_RING_COMPACT", 1) != 0;
  for (int g = 0; g < e->n_groups; ++g) {
    const long long n0 = e->gstart[g], n1 = e->gstart[g + 1];
    bool compact = false;
    if (may_compact) {
      int entry;
      const int series = (int)((e->gseries[g] - e->series) / (2 * (size_t)e->nrows));
      const int st = replay_series_entry(a->replay, e->serial, series, e->gseries[g], e->nrows, e->stream, &entry);
      if (st) return st;
      compact = entry >= 0;
      S.src_entry = compact ? ring_tag(entry, 0) : 0u;
    }
    const bool lean = may_lean && e->gdp[g].fast_all && (!a->replay || (compact && e->n % 32 == 0 && S.cap % 32 == 0));
    const bool pair = lean && e->uniform_row && pair_mode != 0 && (n1 - n0) % 2 == 0 && (!a->replay || (S.head + n0) % 2 == 0) &&
                      rollout_pair_fills(e->device, n1 - n0, pair_mode);
    const int mb = rollout_min_blocks(e->device, n1 - n0, compact, lean);
    COUNT_LAUNCH();
    if (pair) __atomic_add_fetch(&g_pair_launches, 1, __ATOMIC_RELAXED);
    switch (a->policy) {
      case SHEMS_POLICY_RULE: launch_rollout<SHEMS_POLICY_RULE>(e, a, S, keys, lockstep, g, pair, lean, compact, mb); break;
      case SHEMS_POLICY_RANDOM: launch_rollout<SHEMS_POLICY_RANDOM>(e, a, S, keys, lockstep, g, pair, lean, compact, mb); break;
      default: launch_rollout<SHEMS_POLICY_TAPE>(e, a, S, keys, lockstep, g, pair, lean, compact, mb); break;
    }
  }
  CUDA_TRY(cudaGetLastError());
  e->max_idx += a->n_steps;
  e->step += a->n_steps;
  e->consistent = true;
  if (a->replay) return replay_after_rollout(a->replay, total, e->n, e->stream);   // step t of instance i went to slot head + t*n + i
  return SHEMS_OK;
}
