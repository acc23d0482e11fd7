// shems_device.cuh — the shems_LU1 transition as straight-line device code.
//
// Reference: RL-SHEMS/RL_environments/envs/shems_LU1.jl — action(env, a) :283-316,
// action(env, track) :318-340, step! :343-485, next_state! :264-281.
//
// The Julia source is dynamically typed: which intermediates are Float32 and which are Float64
// depends on the branch (zeros(11) are Float64, b.rate_max is Float64, `pv_ = 0` is an Int ...).
// Here the flow branches are evaluated with predicates/selects into a canonical set of registers —
// doubles holding exactly-representable Float32 or genuine Float64 values — and the common tail
// applies the rounding each branch implies; the two branches whose partial sums stay Float32 in Julia
// (A2a: PV_EV + B_EV, B1a: B_DE + B_EV) are flagged.  Built with -fmad=false: Julia never contracts
// a*b+c, so neither may this file (explicit fma()/fmaf() calls below are the only fused ops).
#pragma once
#include "common.h"

struct StepIn {
  float Soc_b, Soc_ev, c_ev, d_e, g_e, p_buy;
};
struct StepOut {
  float Soc_b, Soc_ev;  // endogenous part of s' (before next_state! overrides Soc_ev on arrival)
  double reward;        // env.reward (Float64)
};
struct StepTrace {  // the remaining `results` columns (:476-478); all values exact in double
  double EV, profit, discomfort, penalty, PV_DE, B_DE, GR_DE, PV_B, PV_GR, PV_EV, B_EV, GR_EV, EX_EV, B;
};

// one 32-byte series row (env.cu: the series layout)
struct Row8 { float soc_ev, cd, d_e, g_e, p_buy, h_cos, h_sin, season; };
__device__ __forceinline__ Row8 load_row(const float4* __restrict__ series, int row1 /*1-based*/) {
  const float4 a = __ldg(series + 2 * (size_t)(row1 - 1));
  const float4 b = __ldg(series + 2 * (size_t)(row1 - 1) + 1);
  Row8 r;
  r.soc_ev = a.x; r.cd = a.y; r.d_e = a.z; r.g_e = a.w; r.p_buy = b.x; r.h_cos = b.y; r.h_sin = b.z; r.season = b.w;
  return r;
}

__device__ __forceinline__ float jl_minf(float x, float y) { return (y < x) ? y : x; }     // Base.min(x, y), no NaN
__device__ __forceinline__ double jl_mind(double x, double y) { return (y < x) ? y : x; }
// Base.clamp(x, lo, hi) = ifelse(x > hi, hi, ifelse(x < lo, lo, x))
__device__ __forceinline__ double jl_clampd(double x, double lo, double hi) { return (x > hi) ? hi : ((x < lo) ? lo : x); }

// IEEE-754 correctly rounded x / d for a CONSTANT divisor as q = x*r; e = x - q*d (exact, FMA); q' = q + e*r.
// Float32: `ok` says the host verified the sequence against x/d for all 2^23 significands of this d
// (env.cu: verify_fdiv_const); operands so small that the residual would be subnormal take the IEEE path.
__device__ __forceinline__ float fdiv_const(float x, float d, float r, int ok) {
  if (!ok || (fabsf(x) < 8.6736174e-19f /* 2^-60 */ && x != 0.0f)) return x / d;
  const float q = x * r;
  const float e = fmaf(-q, d, x);
  return fmaf(e, r, q);
}
// The same Float32 quotient through Float64, branch-free and without a guard: RN32(RN64(x / d)) == RN32(x / d) for every pair of
// Float32 operands (double rounding is innocuous for division once the wide format has >= 2p + 2 = 50 significant bits), and
// RN64(x / d) is what ddiv_const (below) delivers for a Float32-valued constant divisor.  Every Float32 — subnormals included — is
// a normal double, so no operand needs the IEEE fallback; x = 0 gives 0.  xd = (double)x is passed in because the callers need it anyway.
__device__ __forceinline__ double ddiv_const(double x, double d, double r, int ok);
__device__ __forceinline__ float fdiv_const_wide(double xd, double d_d, double r_d) {
  const double q = xd * r_d;
  const double e = fma(-q, d_d, xd);
  return (float)fma(e, r_d, q);
}
// Float64 with a divisor that is a converted Float32 (<= 24 significant bits): q + e*r differs from x/d by
// < 2^-105 relative, while x/d is either exactly representable-or-farther than 2^-77 relative from any
// rounding midpoint (x - m*d lies on a grid of 2^-76 |x| and cannot vanish for a 54-bit odd m), so
// RN(q + e*r) == RN(x/d) for every normal x.  `ok` = the divisor really is Float32-valued.
__device__ __forceinline__ double ddiv_const(double x, double d, double r, int ok) {
  if (!ok) return x / d;
  const double q = x * r;
  const double e = fma(-q, d, x);
  return fma(e, r, q);
}

// Row class: the values of the step's predicates that depend only on the series row — A = Float32(g_e * pv_eta) > d_e (PV covers the
// demand, :368), c_ev > -1 (EV present, :292), c_ev == 0 (departure hour, :438), c_ev < 0 (no EV, :445) and c_ev == -1 (arrival test,
// :270).  ROW_ANY evaluates them at run time; every other class fixes them, so a body instantiated for it is the same code with those
// predicates as constants.  row_class() derives the class from the very expressions the step evaluates, so a lane gets the same bits
// from the body of its class as from the ROW_ANY body.  Departure hours, -0.0, values in (-1, 0) and NaN stay ROW_ANY.
enum RowClass { ROW_ANY = 0, ROW_A_NOEV, ROW_B_NOEV, ROW_A_EV, ROW_B_EV };   // A / B: branch :368 / :388; NOEV: c_ev == -1; EV: c_ev > 0
__device__ __forceinline__ int row_class(const DevParams& P, float c_ev, float d_e, float g_e) {
  const bool A = g_e * P.pv_eta > d_e;
  if (c_ev == -1.0f) return A ? ROW_A_NOEV : ROW_B_NOEV;
  if (c_ev > 0.0f) return A ? ROW_A_EV : ROW_B_EV;
  return ROW_ANY;
}
// what a class other than ROW_ANY fixes; the step writes each predicate as `CLS == ROW_ANY ? <run-time test> : <constant>` in place
template <int CLS> constexpr bool row_A = CLS == ROW_A_NOEV || CLS == ROW_A_EV;         // A
template <int CLS> constexpr bool row_ev = CLS == ROW_A_EV || CLS == ROW_B_EV;          // c_ev > 0: c_ev > -1, not == 0, not < 0, not == -1
template <int CLS> constexpr bool row_noev = CLS == ROW_A_NOEV || CLS == ROW_B_NOEV;    // c_ev == -1: not > -1, not == 0, < 0, == -1

// next_state! :264-281: Soc_ev of s' after a step from a row with countdown cd_here (class CLS) to row nx — the row's soc_ev when an
// EV arrives there (:270-272), else the step's own.  nx is taken by value (by reference the lean and pair rollout kernels compile the
// select with its operands swapped) and cd_here by reference (so that actor_rollout_kernel reads it from shared memory only when
// nx.cd >= 0, as it always has).
template <int CLS = ROW_ANY>
__device__ __forceinline__ float next_soc_ev(float step_soc_ev, Row8 nx, const float& cd_here) {
  return (nx.cd >= 0.0f && (CLS == ROW_ANY ? cd_here == -1.0f : row_noev<CLS>)) ? nx.soc_ev : step_soc_ev;
}

// FAST (template parameter of everything below) = the constants are in their usual state — P.fast_all: Float32-valued divisors,
// Float32 penalty weight, shems_LU1's reward form — so the flag tests, the fall-back branches and the guarded Float32 division
// sequences are compiled out (the Float32 quotients go through fdiv_const_wide), and Float32 decisions against Float64 constants are
// taken in FP32 against thresholds the host rounded (x > c <=> x > RD32(c), x < c <=> x < RU32(c) for Float32 x; the Float32 value
// of c where a branch yields it is RN32(c)).  Both instantiations give the same bits.

// Float32(clamp(Float64(pv), 0.0, min(R, Float64(h)))) for Float32 pv, h (charge request, :307-308 / :331-332): h < R <=> h < RU32(R),
// pv > R <=> pv > RD32(R), and the Float64 result is h, R, 0 or pv, so its Float32 value is h, RN32(R), 0 or pv
__device__ __forceinline__ float charge_request_f(const DevParams& P, float pv, float h) {
  const bool h_lo = h < P.R_up;
  return (pv > (h_lo ? h : P.R_dn)) ? (h_lo ? h : P.R_f) : ((pv < 0.0f) ? 0.0f : pv);
}
// Float32(-min(R, Float64(x))) for Float32 x (discharge request, :310 / :334): x < R <=> x < RU32(R); -RN32(R) = RN32(-R)
__device__ __forceinline__ float discharge_request_f(const DevParams& P, float x) { return -((x < P.R_up) ? x : P.R_f); }

// action(env, a::ShemsAction) :283-316 -> Float32.([B, EV])
template <bool FAST, int CLS = ROW_ANY>
__device__ __forceinline__ void shems_action_drl(const DevParams& P, float Soc_b, float Soc_ev, float c_ev, float d_e,
                                                 float g_e, float Bt, float EVt, float& B, float& EV) {
  const float sb0 = Soc_b - P.smin;
  const float perc = FAST ? fdiv_const_wide((double)sb0, P.span_d, P.r_span_d) : fdiv_const(sb0, P.span, P.r_span_f, P.fast_span_f);   // :288
  EV = ((CLS == ROW_ANY ? c_ev > -1.0f : row_ev<CLS>) && Soc_ev < EVt) ? jl_minf(P.evR, (EVt - Soc_ev) * P.C) : 0.0f;      // :292-297
  const float pv = (g_e - d_e) - EV;                                                      // :301
  // :304-313 evaluated branch-free: charge request / discharge request / nothing
  const float Btv = Bt * P.span + P.smin;                                                 // :306 (two roundings, fmad off)
  float Bc, Bd;
  if (FAST) {
    Bc = charge_request_f(P, pv, (Btv - Soc_b) + P.loss);
    Bd = discharge_request_f(P, P.one_m_l * Soc_b);
  } else {
    const double hi = jl_mind(P.R, (double)((Btv - Soc_b) + P.loss));                     // :307
    Bc = (float)jl_clampd((double)pv, 0.0, hi);
    Bd = (float)(-jl_mind(P.R, (double)(P.one_m_l * Soc_b)));                             // :310
  }
  B = (pv > 0.0f && perc < Bt) ? Bc : ((Soc_b > 1e-3f) ? Bd : 0.0f);
}

// action(env, track) rule-based controller :318-340 -> Float32.([B, EV]); it reads no row predicate, so it takes no row class
template <bool FAST>
__device__ __forceinline__ void shems_action_rule(const DevParams& P, float Soc_b, float Soc_ev, float d_e, float g_e,
                                                  float& B, float& EV) {
  EV = jl_minf(P.evR, (1.0f - Soc_ev) * P.C);                                     // :323
  const float pv = (g_e - d_e) - EV;                                              // :327
  if (FAST) {
    const float Bc = charge_request_f(P, pv, (P.smax - Soc_b) + P.loss);
    const float Bd = discharge_request_f(P, P.one_m_l * Soc_b);
    B = (pv > 0.0f && Soc_b < P.smax95_up) ? Bc : ((Soc_b > 1e-3f) ? Bd : 0.0f);   // Soc_b < 0.95 smax <=> Soc_b < RU32(0.95 smax)
    return;
  }
  const double hi = jl_mind(P.R, (double)((P.smax - Soc_b) + P.loss));            // :331
  const float Bc = (float)jl_clampd((double)pv, 0.0, hi);
  const float Bd = (float)(-jl_mind(P.R, (double)(P.one_m_l * Soc_b)));           // :334
  B = (pv > 0.0f && (double)Soc_b < P.smax95) ? Bc : ((Soc_b > 1e-3f) ? Bd : 0.0f);  // :330 (0.95 is Float64), :333
}

// step! :343-485 given the feasible (B, EV) and the recorded EV target.  track_neg <=> track < 0
// (no penalty in the reward, :466-471).
// w * discomfort^pot (shems_LU1 / shems_LU7) or (discomfort * w)^pot (shems_LU1_input0607) for the exponents other than LU1's 2
static __device__ __noinline__ double shems_discomfort_term(int reward_form, double dw, double pot, double dd) {
  if (!reward_form) return dw * ((pot == 2.0) ? dd * dd : (pot == 1.0) ? dd : pow(dd, pot));
  const double dwd = dd * dw;
  return (pot == 1.0) ? dwd : (pot == 2.0) ? dwd * dwd : pow(dwd, pot);
}

template <bool WANT_TRACE, bool FAST, int CLS = ROW_ANY>
__device__ __forceinline__ StepOut shems_flows(const DevParams& P, const StepIn& s, float B, float EV, float EVt,
                                               bool track_neg, StepTrace* tr) {
  const float eta = P.b_eta;
  const double eta_d = P.eta_d;
  // :362-364  battery discharge budget (Float64).  F32 < -0.01 (Float64 literal) <=> F32 < -0.01f0.
  const double BD0 = (B < -0.01f) ? jl_clampd((double)(-B), 0.001, jl_mind(P.R, (double)(P.one_m_l_e * s.Soc_b))) : 0.0;
  // :368-409  PV -> demand -> EV, then battery -> demand -> EV, grid takes the slack
  const float ge = s.g_e * P.pv_eta;
  const bool A = CLS == ROW_ANY ? ge > s.d_e : row_A<CLS>;   // :368 PV covers the demand      (else :388)
  const float pvr = ge - s.d_e;              // :370 PV left after the demand   (branch A)
  const float dB = s.d_e - ge;               // :391 demand left after the PV   (branch B)
  const bool A1 = A && (pvr > EV);           // :371 PV also covers the EV
  const float PV_DE = A ? s.d_e : ge;        // :369 / :389
  const float PV_EV = A ? (A1 ? EV : pvr) : 0.0f;   // :372 / :375
  const float pv = A1 ? (pvr - EV) : 0.0f;   // :373 / :376 / :390  (Float32, or the Int 0)
  // battery stage 1 (branch B only): the residual demand dB   :392-408
  const float q1 = FAST ? fdiv_const_wide((double)dB, eta_d, P.r_eta_d) : fdiv_const(dB, eta, P.r_eta_f, P.fast_eta_f);
  const bool cover1 = (!A) && (BD0 > (double)q1);
  const double B_DE = A ? 0.0 : (cover1 ? (double)dB : BD0 * eta_d);              // :393 / :404
  const double GR_DE = (A || cover1) ? 0.0 : ((double)dB - B_DE);                 // :406
  const double BD1 = A ? BD0 : (cover1 ? BD0 - (double)q1 : 0.0);                 // :394 / :405
  // battery stage 2: the EV share not served by PV — x2 = EV - PV_EV (:377-384); in branch B it is EV itself (:395-402)
  const float x2 = EV - PV_EV;
  const float q2 = FAST ? fdiv_const_wide((double)x2, eta_d, P.r_eta_d) : fdiv_const(x2, eta, P.r_eta_f, P.fast_eta_f);
  const bool act2 = A ? (!A1) : cover1;
  const bool cover2 = act2 && (BD1 > (double)q2);
  const double B_EV = cover2 ? (double)x2 : (act2 ? BD1 * eta_d : 0.0);           // :378/:396, :381/:399
  const double GR_EV = cover2 ? 0.0 : (act2 ? ((double)x2 - B_EV) : (A ? 0.0 : (double)EV));  // :383/:401, :407
  // Julia keeps these two partial sums in Float32 (both addends are Float32 on exactly these paths)
  const bool leafA2a = A && cover2;          // PV_EV + B_EV  (:435)
  const bool leafB1a = (!A) && cover2;       // B_DE + B_EV   (:432)
  const float f32sum = A ? (PV_EV + x2) : (dB + EV);
  // :412-422 battery charging.  F32 > 0.01 (Float64) <=> F32 > 0.01f0
  double PV_B = 0.0, X = (double)s.Soc_b, pv_d = (double)pv;
  if (B > 0.01f) {
    const double BC = jl_clampd((double)B, 0.001, jl_mind(P.R, (double)(P.smax - s.Soc_b)));   // :413
    const double thr = ddiv_const(BC, eta_d, P.r_eta_d, FAST ? 1 : P.fast_d);
    const bool c1 = pv_d > thr;              // :414
    const float pvb = pv * eta;              // :418 stays Float32 (pv_ is Float32 or the Int 0)
    PV_B = c1 ? BC : (double)pvb;
    X = c1 ? ((double)s.Soc_b + BC) : (double)(s.Soc_b + pvb);
    pv_d = c1 ? (pv_d - thr) : 0.0;          // :416 / :419
  }
  // :432  (1 - loss) * (Soc_b + PV_B + GR_B - (B_DE + B_EV + B_GR) / eta)
  double Y = 0.0;
  if (BD0 > 0.0) {  // without a discharge budget B_DE = B_EV = 0 and the quotient is 0
    const double Yd = ddiv_const(B_DE + B_EV, eta_d, P.r_eta_d, FAST ? 1 : P.fast_d);
    const float Yf = FAST ? fdiv_const_wide((double)f32sum, eta_d, P.r_eta_d) : fdiv_const(f32sum, eta, P.r_eta_f, P.fast_eta_f);
    Y = leafB1a ? (double)Yf : Yd;
  }
  StepOut o;
  o.Soc_b = (float)(P.one_m_l_d * (X - Y));
  // :435  Soc_ev + (PV_EV + B_EV + GR_EV) / (ev.soc_max - ev.soc_min)
  const double T = leafA2a ? (double)f32sum : (((double)PV_EV + B_EV) + GR_EV);
  float Soc_ev_new = s.Soc_ev;
  if (T != 0.0) Soc_ev_new = (float)((double)s.Soc_ev + ddiv_const(T, P.C_d, P.r_C_d, FAST ? 1 : P.fast_d));
  // :438-449
  float disc = 0.0f, EX_EV = 0.0f;
  double pen = 0.0;
  if ((CLS == ROW_ANY ? s.c_ev == 0.0f : false) && Soc_ev_new < 1.0f) {
    const float short_ = 1.0f - Soc_ev_new;
    disc = short_ * 100.0f;
    EX_EV = short_ * P.C;
    Soc_ev_new = 1.0f;
  } else if ((CLS == ROW_ANY ? s.c_ev < 0.0f : row_noev<CLS>) && EVt < 0.99f) {  // F32 < 0.99 (Float64) <=> F32 < 0.99f0
    // shems_LU1: Float32 product with penalty_weight::Float32; LU7 / input0607: penalty_weight is a Float64 -> Float64 product
    const float om = 1.0f - EVt;
    pen = (double)(om * P.pw);
    if (!FAST && P.pen_f64) pen = (double)om * P.pw_d;
  }
  o.Soc_ev = Soc_ev_new;
  // :464  profit = (sell * p_buy * (PV_GR + B_GR)) - (p_buy * (GR_DE + GR_B + GR_EV + EX_EV))   [Float64]
  const double pb = (double)s.p_buy;
  const double profit = ((P.sell * pb) * pv_d) - (pb * ((GR_DE + GR_EV) + (double)EX_EV));
  const double dd = (double)disc;
  // Float32^Float64 promotes; x*x is exact for F32 x, x^1.0 is x
  double dterm = P.dw * (dd * dd);                                   // reward_mode 0: shems_LU1's w * discomfort^2
  if (!FAST && P.reward_mode != 0) dterm = shems_discomfort_term(P.reward_form, P.dw, P.pot, dd);      // every other combination (uniform branch, off the hot path)
  const double base = profit - dterm;
  if (track_neg) pen = 0.0;  // :466-468
  o.reward = track_neg ? base : (base - pen);
  if (WANT_TRACE) {
    tr->EV = (double)EV; tr->profit = profit; tr->discomfort = dd; tr->penalty = pen;
    tr->PV_DE = (double)PV_DE; tr->B_DE = B_DE; tr->GR_DE = GR_DE; tr->PV_B = PV_B; tr->PV_GR = pv_d;
    tr->PV_EV = (double)PV_EV; tr->B_EV = B_EV; tr->GR_EV = GR_EV; tr->EX_EV = (double)EX_EV; tr->B = (double)B;
  }
  return o;
}

// the `results` row :476-478 of a step from row idx, column c at q[c * N]
__device__ __forceinline__ void store_trace_row(double* __restrict__ q, long long N, int idx, const StepIn& s, float Bt, float EVt,
                                                const StepOut& o, const StepTrace& tr) {
  q[SHEMS_T_INDEX * N] = (double)(idx + 1); q[SHEMS_T_C_EV * N] = (double)s.c_ev; q[SHEMS_T_EV_TARGET * N] = (double)EVt;
  q[SHEMS_T_EV * N] = tr.EV; q[SHEMS_T_SOC_EV * N] = (double)s.Soc_ev; q[SHEMS_T_REWARD * N] = o.reward;
  q[SHEMS_T_PROFIT * N] = tr.profit; q[SHEMS_T_DISCOMFORT * N] = tr.discomfort; q[SHEMS_T_PENALTY * N] = tr.penalty;
  q[SHEMS_T_PV_DE * N] = tr.PV_DE; q[SHEMS_T_B_DE * N] = tr.B_DE; q[SHEMS_T_GR_DE * N] = tr.GR_DE; q[SHEMS_T_PV_B * N] = tr.PV_B;
  q[SHEMS_T_PV_GR * N] = tr.PV_GR; q[SHEMS_T_PV_EV * N] = tr.PV_EV; q[SHEMS_T_B_EV * N] = tr.B_EV; q[SHEMS_T_GR_EV * N] = tr.GR_EV;
  q[SHEMS_T_EX_EV * N] = tr.EX_EV; q[SHEMS_T_GR_B * N] = 0.0; q[SHEMS_T_B_GR * N] = 0.0; q[SHEMS_T_B * N] = tr.B;
  q[SHEMS_T_B_TARGET * N] = (double)Bt; q[SHEMS_T_SOC_B * N] = (double)s.Soc_b;
}

// env.state of instance n into the structure-of-arrays obs [9][N]: (Soc_b, Soc_ev) and the exogenous fields of series row r
__device__ __forceinline__ void store_obs(float* __restrict__ obs, long long N, long long n, float Soc_b, float Soc_ev, const Row8& r) {
  obs[0 * N + n] = Soc_b; obs[1 * N + n] = Soc_ev; obs[2 * N + n] = r.cd; obs[3 * N + n] = r.d_e; obs[4 * N + n] = r.g_e;
  obs[5 * N + n] = r.p_buy; obs[6 * N + n] = r.h_cos; obs[7 * N + n] = r.h_sin; obs[8 * N + n] = r.season;
}
