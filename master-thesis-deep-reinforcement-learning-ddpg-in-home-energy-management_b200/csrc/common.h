// common.h — internals shared by the translation units of libshems_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/shems_b200.h"
#include "ring.cuh"  // the replay ring's record format and sampling rule

// thread-local last-error string (shems_last_error)
void shems_set_error(const char* fmt, ...);

#define CUDA_TRY(expr)                                                                     \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      shems_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return SHEMS_ERR_CUDA;                                                               \
    }                                                                                      \
  } while (0)

#define REQUIRE(cond, code, ...)  \
  do {                            \
    if (!(cond)) {                \
      shems_set_error(__VA_ARGS__); \
      return (code);              \
    }                             \
  } while (0)

// RAII device guard: every entry point runs on its handle's device and restores the caller's
struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define GUARD(dev)                                             \
  DeviceGuard _guard(dev);                                     \
  if (!_guard.ok) {                                            \
    cudaError_t _e = cudaGetLastError();                       \
    shems_set_error("cannot select CUDA device %d: %s", (dev), cudaGetErrorString(_e)); \
    return SHEMS_ERR_CUDA;                                     \
  }

// constants of the env with the derived values every step needs (passed by value to kernels)
struct DevParams {
  float pv_eta, b_eta, smin, smax, loss, evmin, evmax, evR, pw;
  float one_m_l;     // Float32(1 - b.loss)
  float one_m_l_e;   // Float32(Float32(1 - b.loss) - 1f-7)
  float C;           // ev.soc_max - ev.soc_min
  float span;        // b.soc_max - b.soc_min
  float R_f;         // Float32(b.rate_max) = RN32(R)
  float R_dn, R_up;  // RD32(R), RU32(R): Float32 comparisons with R (FAST: charge_request_f / discharge_request_f)
  float smax95_up;   // RU32(smax95)
  double R, sell, dw, pot;
  double pw_d;               // Float64 penalty weight of the sibling envs (pen_f64 != 0)
  int pen_f64, reward_form;
  int reward_mode;           // 0: w*discomfort^2 in form 0 (shems_LU1, the fast path); 1: anything else (shems_discomfort_term)
  double eta_d, one_m_l_d, C_d, smax95;
  // division by the constants eta / span / C as multiply + 2 FMA (see fdiv_const / ddiv_const in shems_device.cuh)
  float r_eta_f, r_span_f;   // Float32(1/eta), Float32(1/span)
  double r_eta_d, r_C_d;     // 1/Float64(eta), 1/Float64(C)
  int fast_eta_f, fast_span_f;  // host-verified over all 2^23 significands: the 3-op sequence == IEEE division
  int fast_d;                   // eta_d and C_d are Float32-valued: the 3-op sequence is provably correctly rounded
  double span_d, r_span_d;      // Float64(span), 1/Float64(span): the Float32 quotient Soc_b / span through Float64 (fdiv_const_wide)
  int fast_all;                 // fast_d && span Float32-valued && Float32 penalty weight && shems_LU1's reward form: kernels take the
                                // FAST instantiation (no flag tests, no guarded division sequences) — same results
};

#define SHEMS_MAX_GROUPS 16

struct RingSeries {                // the ring's copy of one env series
  unsigned long long env_serial;   // ShemsEnv::serial of the env it was copied from (never a pointer: those get reused after free)
  int series;                      // which of that env's series (0 when the groups share one)
  int nrows;
  float* rows;                     // device, nrows x 8 floats
};

struct ShemsReplay {
  int device;
  cudaStream_t stream;
  int64_t capacity, length, head;  // head = physical slot of the next push
  float* alloc;  // the series-table header + the ring (ring_alloc_floats)
  float* ring;   // ring_in_alloc(alloc): tiled SoA, see ring.cuh: ceil(cap/32) tiles x 23 fields x 32 slots
  int32_t* idx_scratch;  // device scratch for sampled indices
  int64_t idx_scratch_n;
  float* minmax_scratch; // [18]
  void* group_refs; int group_refs_n;  // device scratch of replay_push_groups (ring / capacity / head of every learner's memory)
  RingSeries src[RING_MAX_SERIES];     // series table of the compact records (entry i <-> header pointer i)
  const float* src_ptrs[RING_MAX_SERIES];
  int n_src;
  float* prio_alloc;  // replay_enable_priorities: header + sum tree of the slots' priorities (ring.cuh), else NULL
  float* prio;        // node 0 of the tree (prio_alloc + PRIO_HEADER_FLOATS)
  int64_t prio_p2;    // prio_p2(capacity)
  int32_t* next;      // replay_enable_successors: next[cap], the successor link of every slot (ring.cuh), else NULL
};

struct ShemsEnv {
  int device;
  cudaStream_t stream;
  DevParams dp;
  ShemsParams params;
  int32_t nrows, maxsteps;
  int64_t n;
  float4* series;   // [nrows][2] rows: (soc_ev, h_countdown, electkwh, PV_generation | p_buy, hour_cos, hour_sin, season)
  float* obs;       // [9][n]  == env.state of every instance
  int32_t* idx;     // [n] 1-based row (env.idx)
  int32_t* d_maxidx;  // device scalar: max idx after reset
  int32_t max_idx;    // host mirror: the largest row any instance is on, or (while max_pending) an upper bound of it; +1 per step
  int32_t* h_maxidx;  // pinned host word the reset kernel's maximum is copied to (asynchronously)
  cudaEvent_t ev_maxidx; bool max_pending;  // the exact value is fetched only when the upper bound does not settle a bounds check
  int32_t step;       // env.step (instances run in lockstep)
  unsigned long long serial;  // unique per env handle of the process (keys the replay rings' series tables)
  bool was_reset;
  bool consistent;    // state fields 2..8 equal series row idx (false after shems_set_state)
  bool uniform_row;   // every instance stands on the same row (steps keep it: each instance advances one row per step); like
                      // `consistent`, writes through shems_state_ptr must keep it true
  int32_t* scratch_i; float* scratch_f; // staging for reset host draws
  // groups of instances with their own constants (several chargers in one handle): group g = instances gstart[g] .. gstart[g+1]-1
  int n_groups;
  DevParams gdp[SHEMS_MAX_GROUPS];
  float4* gseries[SHEMS_MAX_GROUPS];
  long long gstart[SHEMS_MAX_GROUPS + 1];
};

// a writer has stored n_written transitions from slot head on, `width` instances per step (slot head + t*width + i holds step t of
// instance i): advances head and length, and enqueues on `st` (the writer's stream, after the records are written) the refresh that
// gives the surviving min(n_written, cap) slots the priority p_max (a memory with priorities) and the successor-link pass over them
// (a memory with links)
int replay_after_rollout(ShemsReplay* rp, int64_t n_written, int64_t width, cudaStream_t st);
// entry of rp's series table holding series `series` of env `serial` (nrows rows at rows_dev), copied on first use; -1 when the table
// is full.  The copy is enqueued on rp->stream and `user` (the stream of the writer) waits for it.
int replay_series_entry(ShemsReplay* rp, unsigned long long serial, int series, const float4* rows_dev, int nrows, cudaStream_t user,
                        int* entry);
// may every instance advance `need` more rows (next_state! reads row idx+1)?  0 = yes, else the furthest instance's row (env.cu)
int32_t ensure_rows(ShemsEnv* e, int64_t need);
