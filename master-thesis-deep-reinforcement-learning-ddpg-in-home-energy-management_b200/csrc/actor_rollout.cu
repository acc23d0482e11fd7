// actor_rollout.cu — episode!(env; train = false) and inference(env; track = 1) (RL-SHEMS/algorithms/DDPG.jl:186-242 with
// train == false, src/memory_plotting_saving.jl:62-89) as ONE persistent thread-block-cluster kernel: act(normalize(s)) ->
// scale_action -> step! for T steps without leaving the chip.
//
// The reference evaluates a trained actor one state at a time: per step an actor forward pass on the GPU, a device-to-host copy,
// step! on the host (with its CSV parse), 1439 / 2999 / 4319 times for an inference run and 100 x 72 times for every evaluation
// inside run_episodes (DDPG.jl:266-279).  Here a cluster of 8 CTAs owns 8 instances: each CTA keeps its 250 x 64 slice of the
// actor's W2 in shared memory for the WHOLE episode (staged once), layer 1 is recomputed by every CTA, the output layer's partial
// dot products are all-gathered through distributed shared memory (one cluster barrier per step), and then EVERY CTA advances
// the 8 environment instances redundantly with the Julia-exact transition of shems_device.cuh — identical inputs give
// identical states in all 8 CTAs, so no second exchange is needed; CTA 0 writes the trace rows.
//
// Compiled with -fmad=false like env.cu (the transition restates Julia scalar arithmetic); the network pieces use explicit
// fmaf() and give the bits of csrc/ddpg_fused.cu's act kernel.
#include "ddpg_fused_dev.cuh"
#include "shems_device.cuh"

template <bool WANT_TRACE>
__global__ void __cluster_dims__(FUSED_CLUSTER, 1, 1) __launch_bounds__(FT, 1)
actor_rollout_kernel(const ActorRolloutArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FusedSmem* S = reinterpret_cast<FusedSmem*>(smem_raw);
  __shared__ int s_idx[FUSED_ROWS];
  __shared__ float s_cd[FUSED_ROWS];     // df[env.idx, :h_countdown] of the row the instance stands on (shems_LU1.jl:270)
  __shared__ double s_ret[FUSED_ROWS];   // reward_eps (DDPG.jl:223)
  cg::cluster_group cluster = cg::this_cluster();
  const int tid = threadIdx.x, lane = tid & 31;
  const Geo g = make_geo(a.l1, a.l2, a.vec16, cluster);
  const int l1 = a.l1, l2 = a.l2;
  const long long N = a.N;
  // The launch's instances n0 .. n1-1 are segments of a.seg instances; segment s is learner a.l0 + s and takes ceil(seg / 8)
  // clusters, the rows past its end idle.  One learner: a single segment over the whole range (l0 = 0).
  const long long cps = (a.seg + FUSED_ROWS - 1) / FUSED_ROWS, c = blockIdx.x / FUSED_CLUSTER, sg = c / cps;
  const long long j0 = a.n0 + sg * a.seg + (c - sg * cps) * FUSED_ROWS;   // first instance of this cluster
  const long long jend = a.n0 + (sg + 1) * a.seg;                          // end of its learner's instances
  const float* actor = a.actor + (a.l0 + sg) * a.actor_stride;
  const float* norm = a.norm + (a.l0 + sg) * a.norm_stride;
  float* raw = S->x[1];                  // env.state of the 8 instances [row][12]
  cluster_arrive();
  stage_w2(S->W[0], actor + a.ao.w2, l1, l2, g.n0, g.nv, a.vec16 != 0, tid);
  if (tid < 72) {
    const int r = tid / 9, k = tid - r * 9;
    const long long j = j0 + r;
    raw[r * 12 + k] = (j < jend) ? a.obs[(long long)k * N + j] : 0.0f;
  } else if (tid >= 96 && tid < 96 + FUSED_ROWS) {
    const int r = tid - 96;
    const long long j = j0 + r;
    const int idx = (j < jend) ? a.idx[j] : 1;
    s_idx[r] = idx;
    s_cd[r] = __ldg(&reinterpret_cast<const float*>(a.series)[8 * (size_t)(idx - 1) + 1]);
    s_ret[r] = 0.0;
  }
  const L1Regs Ra = load_l1(actor + a.ao.w1, actor + a.ao.b1, 9, l1, tid);
  const TailRegs Ta = load_tail(actor + a.ao.b2 + g.n0, actor + a.ao.w3 + g.n0 * 2, 2, g.nv, lane);
  const float b3a0 = __ldg(actor + a.ao.b3), b3a1 = __ldg(actor + a.ao.b3 + 1);
  float nlo = 0.0f, nden = 1.0f;         // normalize(): thread (row, field k) keeps its s_min[k] and s_max[k] - s_min[k] + 1f-8
  if (tid < 72) {
    const int k = tid % 9;
    nlo = norm[k];
    nden = __fadd_rn(__fsub_rn(norm[9 + k], nlo), 1e-8f);
  }
  cp_wait<0>();
  __syncthreads();
  cluster_wait();   // every CTA of the cluster runs: its shared memory may be written from now on
  for (int t = 0; t < a.T; ++t) {
    if (tid < 72) {  // normalize(s) = (s - s_min) / (s_max - s_min + 1f-8)   (memory_plotting_saving.jl:55-57); idle rows stay zero
      const int r = tid / 9, k = tid - r * 9;
      S->x[0][r * 12 + k] = (j0 + r < jend) ? __fdiv_rn(__fsub_rn(raw[r * 12 + k], nlo), nden) : 0.0f;
    }
    __syncthreads();
    f1(Ra, 9, l1, S->x[0], S->h1T[0], tid);
    __syncthreads();
    f2(S->W[0], Ta, l1, g.nv, S->h1T[0], S->red, S->h2s[0], tid);
    const int buf = t & 1;   // two all-gather buffers alternate: a peer refills one only after the barrier that follows my reads of it
    f3_partial(Ta, S->h2s[0], S, buf, cluster, g.rank, tid);
    cluster.sync();
    if (tid < FUSED_ROWS && j0 + tid < jend) {
      const int r = tid;
      const long long j = j0 + r;
      const float y0 = tanhf(xch_sum(S, buf, r, 0) + b3a0), y1 = tanhf(xch_sum(S, buf, r, 1) + b3a1);
      const long long step = (long long)a.step0 + t + 1;
      const unsigned long long rng_step = (a.seed * 1000003ull + (unsigned long long)step) & 0x7fffffffffffffffull;   // as ddpg_episode
      const ActOut o = act_gauss_epilogue(y0, y1, false, 0.0f, 0.0f, a.sigma, rng_step, step, a.env_id_base + j, a.lo0, a.lo1, a.hi0, a.hi1);
      // step!(env, s, scaled_action; track)  (shems_LU1.jl:343-485)
      StepIn s;
      s.Soc_b = raw[r * 12 + 0]; s.Soc_ev = raw[r * 12 + 1]; s.c_ev = raw[r * 12 + 2]; s.d_e = raw[r * 12 + 3]; s.g_e = raw[r * 12 + 4];
      s.p_buy = raw[r * 12 + 5];
      float B, EV;
      shems_action_drl<false>(a.P, s.Soc_b, s.Soc_ev, s.c_ev, s.d_e, s.g_e, o.s0, o.s1, B, EV);
      StepTrace tr;
      const StepOut so = shems_flows<WANT_TRACE, false>(a.P, s, B, EV, o.s1, false, &tr);
      const int idx = s_idx[r];
      const Row8 nx = load_row(a.series, idx + 1);   // next_state! :264-281
      const float Soc_ev_new = next_soc_ev(so.Soc_ev, nx, s_cd[r]);
      if (g.rank == 0) {
        if (WANT_TRACE) store_trace_row(a.trace + (size_t)t * SHEMS_TRACE_COLS * N + j, N, idx, s, o.s0, o.s1, so, tr);
        if (a.act_traj) { a.act_traj[((size_t)t * 2 + 0) * N + j] = o.a0; a.act_traj[((size_t)t * 2 + 1) * N + j] = o.a1; }
      }
      raw[r * 12 + 0] = so.Soc_b; raw[r * 12 + 1] = Soc_ev_new; raw[r * 12 + 2] = nx.cd; raw[r * 12 + 3] = nx.d_e; raw[r * 12 + 4] = nx.g_e;
      raw[r * 12 + 5] = nx.p_buy; raw[r * 12 + 6] = nx.h_cos; raw[r * 12 + 7] = nx.h_sin; raw[r * 12 + 8] = nx.season;
      s_cd[r] = nx.cd;
      s_idx[r] = idx + 1;
      s_ret[r] += so.reward;   // reward_eps += r, Float64 (DDPG.jl:223)
    }
    __syncthreads();
  }
  if (g.rank == 0) {
    if (tid < 72) {
      const int r = tid / 9, k = tid - r * 9;
      if (j0 + r < jend) a.obs[(long long)k * N + j0 + r] = raw[r * 12 + k];
    } else if (tid >= 96 && tid < 96 + FUSED_ROWS) {
      const int r = tid - 96;
      if (j0 + r < jend) {
        a.idx[j0 + r] = s_idx[r];
        if (a.ep_return) a.ep_return[j0 + r] = s_ret[r];
      }
    }
  }
}

int actor_rollout_prepare() {
  CUDA_TRY(cudaFuncSetAttribute(actor_rollout_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FusedSmem)));
  CUDA_TRY(cudaFuncSetAttribute(actor_rollout_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FusedSmem)));
  return SHEMS_OK;
}
int actor_rollout_launch(cudaStream_t st, const ActorRolloutArgs& a) {
  const long long n = a.n1 - a.n0;
  if (n <= 0) return SHEMS_OK;
  if (a.seg < 1 || n % a.seg != 0) { shems_set_error("actor_rollout: %lld instances are not whole segments of %lld", n, a.seg); return SHEMS_ERR_INVALID; }
  const unsigned clusters = (unsigned)((n / a.seg) * ((a.seg + FUSED_ROWS - 1) / FUSED_ROWS));
  if (a.trace) actor_rollout_kernel<true><<<clusters * FUSED_CLUSTER, FT, sizeof(FusedSmem), st>>>(a);
  else actor_rollout_kernel<false><<<clusters * FUSED_CLUSTER, FT, sizeof(FusedSmem), st>>>(a);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}
