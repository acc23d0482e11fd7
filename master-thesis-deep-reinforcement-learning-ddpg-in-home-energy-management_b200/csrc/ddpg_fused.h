// ddpg_fused.h — cluster-fused small-batch DDPG update (csrc/ddpg_fused.cu): the reference's own configuration
// (B = 120, 250/500; RL-SHEMS/algorithms/DDPG.jl:121-145) as two thread-block-cluster kernels instead of 19 dependent GEMM launches.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.h"

#define FUSED_CLUSTER 8        // CTAs per cluster (the portable maximum); a cluster owns FUSED_ROWS minibatch rows
#define FUSED_ROWS 8
#define FUSED_MAX_L1 256       // layer widths the kernels' shared-memory plan covers
#define FUSED_MAX_L2 512
#define FUSED_MAX_BATCH 256    // partial-gradient workspace = batch/8 copies of a net

// per-learner hyper-parameters (ddpg_set_hparams).  The kernels of an update read them here, not as launch arguments: the update runs
// as a captured CUDA graph, and a value baked into it would stay stale after a change.
struct DdpgHparams {
  float eta[2];         // ADAM learning rate per optimiser (0 critic, 1 actor), as bp below
  float gamma, tau;     // discount of the TD target, Polyak rate of soft_update!
  float noise_scale;    // exploration noise: σ_eff = RN32(σ of the call × noise_scale)
};

struct DdpgCtrl {  // device-side control block read by the gather kernel (graph replays need no host patching)
  unsigned long long seed;
  unsigned update;      // counts updates; Philox counter for minibatch draws
  int use_idx;          // 1: indices supplied in idx buffer (consumed batch by batch)
  long long len, head, cap;
  int idx_cursor;
  unsigned blocks_done; // last-block-done counter of the final kernel of an update (advances the counters below)
  double bp[2][2];      // βp of Flux.ADAM per optimiser (0 critic, 1 actor): β^t, advanced after every update
  double rc[2][2];      // 1 / (1 - βp): correctly rounded reciprocals of the two bias-correction divisors
  DdpgHparams hp;       // written by the host only (ddpg_create, ddpg_set_hparams); behind the prefix ddpg_episode rewrites by value
  unsigned dp_epoch;    // data-parallel learner: number of gradient exchanges completed (two per update)
  unsigned dp_blocks_done;
  int dp_error;         // set when a peer's signal did not arrive within DP_TIMEOUT_NS
  unsigned dp_ready;    // blocks of the exchange kernel that have pushed their share of this rank's gradient segment
  unsigned dp_abort;    // exchange number block 0 gave up on (every block skips that update: the decision is grid-uniform)
};

struct FusedNetOff { int w1, b1, w2, b2, w3, b3; };  // float offsets of a net's layers inside its flat buffer [W1|b1|W2|b2|W3|b3]
struct FusedArgs {
  const float *actor, *critic, *actor_t, *critic_t;  // flat parameter buffers (Flux layout Wt[in][out] per layer)
  FusedNetOff ao, co;
  int l1, l2, B;
  const float *xs, *xs2;     // [B][11] normalised (s | a) and (s' | .) rows of the gathered minibatch
  float* xspi;               // [B][11] (s | actor(s)): columns 9, 10 are written by the actor pass
  const float *r, *done;     // [B]
  float *q, *y, *qpi;        // [B] critic(s,a), TD target, critic(s, actor(s))  (loss reporting)
  float* part;               // partial gradients of the net this pass differentiates: [B/8][n_params], one copy per cluster
  long long part_stride;     // = n_params of that net
  float inv_batch;           // (γ of the TD target: ctrl->hp.gamma)
  int vec16;                  // W2 rows are 16-byte aligned in both nets: 16-byte staging copies and shared-memory reads (else 4-byte)
  // The critic pass samples and normalises its cluster's 8 transitions itself (what ddpg_gather_kernel does for the tiled path,
  // getData + normalize of src/memory_plotting_saving.jl:31-57) and leaves the (s_n | a) rows in xs for the actor pass.
  const float* const* rings; // replay ring of the learner (device array of pointers, entry 0), or NULL: caller-supplied SoA arrays
  const float *src_s, *src_a, *src_r, *src_s2, *src_d; long long src_ld;   // [9][ld], [2][ld], [ld], [9][ld], [ld] or NULL (done = 0)
  DdpgCtrl* ctrl; const int32_t* idx; const float* norm;
  float* xs_w;               // = xs, written by the critic pass
};
// may this shape run fused?  (widths within the shared-memory plan, whole clusters of 8 rows)
static inline bool ddpg_fused_shape_ok(int B, int l1, int l2) {
  return B >= FUSED_ROWS && B % FUSED_ROWS == 0 && B <= FUSED_MAX_BATCH && l1 >= 1 && l1 <= FUSED_MAX_L1 && l2 >= 1 && l2 <= FUSED_MAX_L2;
}
// act() for a handful of states (the reference's episode loop acts on ONE state per step, DDPG.jl:148-176): normalize + the actor's
// three layers in one cluster kernel, 8 states per cluster; y [n][2] = actor(normalize(s)) before noise
#define FUSED_ACT_MAX_ROWS 64
struct FusedActArgs {
  const float* actor; FusedNetOff ao; int l1, l2, vec16;
  long long n; const float* obs; long long osk;   // state field k of instance j at obs[k*osk + j]
  const float* norm; float* y;                    // y [n][2] (written when a_out is NULL)
  // optional epilogue in the same kernel (act_epilogue.cuh): a = clamp(y + noise, -1, 1), scaled = scale_action(a); component k of
  // instance j at [k*ask + j].  sprev: copy of the raw states [9][osk] for `remember` (the episode loop's s before step!)
  float* a_out; float* scaled_out; const float* noise; long long ask;
  float sigma; unsigned long long seed; long long step, env_id_base; float lo0, lo1, hi0, hi1;
  float* sprev;
  float* noise_acc; int noise_first;             // noise_eps += mean(noise) per instance (DDPG.jl:224), [n]; first: start from 0f0
};
int ddpg_fused_act(cudaStream_t st, const FusedActArgs& a);
int ddpg_fused_prepare();                                    // shared-memory attribute of both kernels on the current device
int ddpg_fused_critic(cudaStream_t st, const FusedArgs& a);  // targets, TD target, critic forward/backward -> part (critic)
int ddpg_fused_actor(cudaStream_t st, const FusedArgs& a);   // actor-loss forward/backward through the critic -> part (actor)

// episode!(env; train = false) / inference(track = 1) for the instances n0 .. n1-1 of an environment handle as one persistent cluster
// kernel (csrc/actor_rollout.cu): act(normalize(s)) -> scale_action -> step! for T steps, 8 instances per cluster.  Populations: the
// range is (n1 - n0) / seg learners of seg instances each, learner l0 + s taking instances n0 + s*seg ..; a cluster serves one learner
// and reads its actor at actor + l*actor_stride and its s_min / s_max at norm + l*norm_stride.  One learner: seg = n1 - n0, l0 = 0.
struct ActorRolloutArgs {
  const float* actor; FusedNetOff ao; int l1, l2, vec16;
  const float* norm;
  long long seg, l0, actor_stride, norm_stride;
  DevParams P; const float4* series;
  long long N, n0, n1;       // SoA stride of the handle's arrays; instance range of this launch (one group of constants)
  float* obs; int32_t* idx;  // env.state [9][N], env.idx [N]: read at the start, written back at the end
  int T, step0;              // steps to take; env.step before the first one (per-step seeds follow ddpg_episode's rule)
  float sigma; unsigned long long seed; long long env_id_base; float lo0, lo1, hi0, hi1;
  double* ep_return;         // [N] reward_eps (Float64) or NULL
  double* trace;             // [T][23][N] `results` rows or NULL
  float* act_traj;           // [T][2][N] the unscaled actions a or NULL
};
int actor_rollout_prepare();
int actor_rollout_launch(cudaStream_t st, const ActorRolloutArgs& a);
