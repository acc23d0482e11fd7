// ddpg_fused.cu — the small-batch DDPG update (RL-SHEMS/algorithms/DDPG.jl replay :121-145, loss_crit :114, loss_act :116-119)
// as TWO thread-block-cluster kernels.
//
// Why: at the reference's B = 120 one replay() is 3.1e8 FLOP (4 µs of fp32 peak) behind 19 DEPENDENT matrix products; launched one
// by one, every product pays a launch, a trip of its operands through L2 and a grid drain (≈ 5 µs each, DESIGN.md §4.4).  The chain
// is only sequential per SAMPLE: rows of the minibatch never meet before the weight gradients are summed.  So a cluster of 8 CTAs
// takes 8 rows through the whole forward and backward chain:
//   * layer widths are split over the cluster's CTAs (CTA c owns 1/8 of the 500 layer-2 units and 1/8 of the 250 layer-1 units);
//   * layer 1 (K = 9 / 11) is recomputed by every CTA — cheaper than exchanging it;
//   * the CTA's 250 x 64 slice of each W2 is staged in shared memory once (16-byte cp.async, overlapped with layer 1) and serves
//     the forward product and the back-propagation through that layer;
//   * what the CTAs owe each other — output-layer partial dot products (8 x 2 numbers) and the partial dX of layer 2 — moves through
//     DISTRIBUTED SHARED MEMORY (st to the peer's smem + barrier.cluster), never through L2;
//   * every cluster writes its 8-row partial of the weight gradients to its own copy in a workspace; the optimiser kernel adds the
//     B/8 copies in a fixed order (deterministic, like everything else here) — the only grid-wide dependency left.
// One update = critic pass (which also samples and normalises its rows of the minibatch), ADAM(critic), actor pass,
// ADAM(actor)+Polyak: 4 launches instead of 21.
// All sums are fp32 in a fixed order; they differ from the tiled-GEMM path only by summation order.
#include "ddpg_fused_dev.cuh"

// ---- critic pass: y = r + γ(1-done) critic_t(s', actor_t(s'));  loss_crit = mse(critic(s,a), y);  partial ∇critic      (DDPG.jl:131-137)
#define FUSED_CRITIC_KERNEL ddpg_fused_critic_kernel
#define FUSED_CRITIC_NSTEP 0
#include "ddpg_fused_critic.cuh"
#undef FUSED_CRITIC_KERNEL
#undef FUSED_CRITIC_NSTEP
// n-step returns (ddpg_set_nstep > 1): the same pass on the walked rows
#define FUSED_CRITIC_KERNEL ddpg_fused_critic_nstep_kernel
#define FUSED_CRITIC_NSTEP 1
#include "ddpg_fused_critic.cuh"
#undef FUSED_CRITIC_KERNEL
#undef FUSED_CRITIC_NSTEP

// ---- actor pass: loss_act = -mean critic(s, actor(s)) with the UPDATED critic; partial ∇actor                          (DDPG.jl:116-119, :140)
__global__ void __cluster_dims__(FUSED_CLUSTER, 1, 1) __launch_bounds__(FT, 1)
ddpg_fused_actor_kernel(const FusedArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FusedSmem* S = reinterpret_cast<FusedSmem*>(smem_raw);
  cg::cluster_group cluster = cg::this_cluster();
  const int tid = threadIdx.x, lane = tid & 31;
  const Geo g = make_geo(a.l1, a.l2, a.vec16, cluster);
  const int l1 = a.l1, l2 = a.l2;
  float* part = a.part + (long long)(blockIdx.x / FUSED_CLUSTER) * a.part_stride;
  const bool vec16 = a.vec16 != 0;   // 16-byte aligned W2 rows: vector staging and vector shared-memory reads
  cluster_arrive();
  // Launched as a programmatic dependent of ADAM(critic): the actor's forward pass does not read the critic and overlaps it.
  stage_w2(S->W[0], a.actor + a.ao.w2, l1, l2, g.n0, g.nv, vec16, tid);
  if (tid < 72) {
    const int r = tid / 9, i = tid - r * 9;
    S->x[0][r * 12 + i] = a.xs[(long long)(g.row0 + r) * 11 + i];   // s_n
  }
  const L1Regs Ra = load_l1(a.actor + a.ao.w1, a.actor + a.ao.b1, 9, l1, tid);
  const TailRegs Ta = load_tail(a.actor + a.ao.b2 + g.n0, a.actor + a.ao.w3 + g.n0 * 2, 2, g.nv, lane);
  const bool colok = (tid & 63) < g.nv;
  const float w3a0 = colok ? __ldg(a.actor + a.ao.w3 + (g.n0 + (tid & 63)) * 2) : 0.0f;       // b3 through the actor: column tid & 63
  const float w3a1 = colok ? __ldg(a.actor + a.ao.w3 + (g.n0 + (tid & 63)) * 2 + 1) : 0.0f;
  const float b3a = __ldg(a.actor + a.ao.b3 + (tid & 1));
  __syncthreads();   // x
  // actor(s_n)
  f1(Ra, 9, l1, S->x[0], S->h1T[0], tid);
  cp_wait<0>();
  __syncthreads();
  f2(S->W[0], Ta, l1, g.nv, S->h1T[0], S->red, S->h2s[0], tid);
  cluster_wait();
  f3_partial(Ta, S->h2s[0], S, 0, cluster, g.rank, tid);
  grid_dependency_wait();   // the critic is updated
  stage_w2(S->W[1], a.critic + a.co.w2, l1, l2, g.n0, g.nv, vec16, tid);
  const L1Regs Rc = load_l1(a.critic + a.co.w1, a.critic + a.co.b1, 11, l1, tid);
  const TailRegs Tc = load_tail(a.critic + a.co.b2 + g.n0, a.critic + a.co.w3 + g.n0, 1, g.nv, lane);
  const float w3c = colok ? __ldg(a.critic + a.co.w3 + g.n0 + (tid & 63)) : 0.0f;             // b3 through the critic
  const float w1a0 = (lane < g.n1v) ? __ldg(a.critic + a.co.w1 + 9 * l1 + g.k0 + lane) : 0.0f;   // critic W1 rows of the two action inputs,
  const float w1a1 = (lane < g.n1v) ? __ldg(a.critic + a.co.w1 + 10 * l1 + g.k0 + lane) : 0.0f;  // this CTA's layer-1 units
  const float b3c = __ldg(a.critic + a.co.b3);
  cluster.sync();
  if (tid < 16) {
    const int r = tid >> 1, j = tid & 1;
    const float pi = tanhf(xch_sum(S, 0, r, j) + b3a);
    S->x[0][r * 12 + 9 + j] = pi;                                   // vcat(s_n, actions)
  }
  __syncthreads();
  // critic(s_n, actor(s_n)), d(-mean q)/dq = -1/B
  f1(Rc, 11, l1, S->x[0], S->h1T[1], tid);
  if (tid < 16) S->dout[tid] = (tid & 1) ? 0.0f : -a.inv_batch;
  cp_wait<0>();
  __syncthreads();
  f2(S->W[1], Tc, l1, g.nv, S->h1T[1], S->red, S->h2s[1], tid);
  f3_partial(Tc, S->h2s[1], S, 1, cluster, g.rank, tid);   // q(s, actor(s)): reporting only
  b3_dz(w3c, 0.0f, 1, g.nv, S->h2s[1], S->dout, S->dzT, tid);
  __syncthreads();
  bx2(S->W[1], S->dzT, l1, g.nv, g.n1s, vec16, S, cluster, g.rank, tid);
  cluster.sync();
  if (tid >= 64 && tid < 72) S->qv[tid - 64] = xch_sum(S, 1, tid - 64, 0) + b3c;
  rs_finish(S, S->h1T[1], g.k0, g.n1v, tid);
  __syncthreads();
  {  // back through critic layer 1 to the two action inputs: this CTA's layer-1 units' share, row = warp
    const int w = tid >> 5;
    const float d = (w < 8) ? S->dz1s[w * 32 + lane] : 0.0f;   // zero beyond the slice; warps 8.. (FT = 512) have no row
    float p0 = w1a0 * d, p1 = w1a1 * d;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { p0 += __shfl_xor_sync(0xffffffffu, p0, o); p1 += __shfl_xor_sync(0xffffffffu, p1, o); }
    if (w < 8 && lane < FUSED_CLUSTER) {
      FusedSmem* peer = cluster.map_shared_rank(S, lane);
      peer->xch[2][(g.rank * 8 + w) * 2 + 0] = p0;
      peer->xch[2][(g.rank * 8 + w) * 2 + 1] = p1;
    }
  }
  cluster.sync();
  if (tid < 16) {  // times tanh'
    const int r = tid >> 1, j = tid & 1;
    const float pi = S->x[0][r * 12 + 9 + j];
    S->dout[r * 2 + j] = xch_sum(S, 2, r, j) * (1.0f - pi * pi);
  }
  __syncthreads();
  // actor backward (global-memory writes after the last cluster barrier, as in the critic pass)
  b3_dz(w3a0, w3a1, 2, g.nv, S->h2s[0], S->dout, S->dzT, tid);
  __syncthreads();
  bx2(S->W[0], S->dzT, l1, g.nv, g.n1s, vec16, S, cluster, g.rank, tid);
  cluster.sync();
  if (g.rank == 0) {
    if (tid < 16) a.xspi[(long long)(g.row0 + (tid >> 1)) * 11 + 9 + (tid & 1)] = S->x[0][(tid >> 1) * 12 + 9 + (tid & 1)];
    else if (tid >= 64 && tid < 72) a.qpi[g.row0 + tid - 64] = S->qv[tid - 64];
  }
  b3_grads(2, g.nv, S->h2s[0], S->dout, part + a.ao.w3 + g.n0 * 2, g.rank == 0 ? part + a.ao.b3 : nullptr, tid);
  bw2(S->h1T[0], S->dzT, l1, l2, g.nv, part + a.ao.w2 + g.n0, part + a.ao.b2 + g.n0, tid);
  rs_finish(S, S->h1T[0], g.k0, g.n1v, tid);
  __syncthreads();
  bw1(S->x[0], 9, S->dz1s, l1, g.n1v, part + a.ao.w1 + g.k0, part + a.ao.b1 + g.k0, tid);
}

// ---- act: y = actor(normalize(s)) for up to 8 states per cluster                                                        (DDPG.jl:148-176)
__global__ void __cluster_dims__(FUSED_CLUSTER, 1, 1) __launch_bounds__(FT, 1)
ddpg_fused_act_kernel(const FusedActArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FusedSmem* S = reinterpret_cast<FusedSmem*>(smem_raw);
  cg::cluster_group cluster = cg::this_cluster();
  const int tid = threadIdx.x, lane = tid & 31;
  const Geo g = make_geo(a.l1, a.l2, a.vec16, cluster);
  const int l1 = a.l1, l2 = a.l2;
  cluster_arrive();
  stage_w2(S->W[0], a.actor + a.ao.w2, l1, l2, g.n0, g.nv, a.vec16 != 0, tid);
  if (tid < 72) {  // normalize(s) = (s - s_min) / (s_max - s_min + 1f-8); rows beyond n are zero
    const int r = tid / 9, k = tid - r * 9;
    const long long j = g.row0 + r;
    float v = 0.0f;
    if (j < a.n) {
      const float lo = a.norm[k];
      const float den = __fadd_rn(__fsub_rn(a.norm[9 + k], lo), 1e-8f);
      const float raw = a.obs[(long long)k * a.osk + j];
      v = __fdiv_rn(__fsub_rn(raw, lo), den);
      if (a.sprev && g.rank == 0) a.sprev[(long long)k * a.osk + j] = raw;
    }
    S->x[0][r * 12 + k] = v;
  }
  const L1Regs Ra = load_l1(a.actor + a.ao.w1, a.actor + a.ao.b1, 9, l1, tid);
  const TailRegs Ta = load_tail(a.actor + a.ao.b2 + g.n0, a.actor + a.ao.w3 + g.n0 * 2, 2, g.nv, lane);
  const float b3a = __ldg(a.actor + a.ao.b3 + (tid & 1));
  __syncthreads();   // x
  f1(Ra, 9, l1, S->x[0], S->h1T[0], tid);
  cp_wait<0>();
  __syncthreads();
  f2(S->W[0], Ta, l1, g.nv, S->h1T[0], S->red, S->h2s[0], tid);
  cluster_wait();
  f3_partial(Ta, S->h2s[0], S, 0, cluster, g.rank, tid);
  cluster.sync();
  if (g.rank == 0 && tid < 16) {
    const int r = tid >> 1, j = tid & 1;
    const long long row = g.row0 + r;
    const float y = tanhf(xch_sum(S, 0, r, j) + b3a);
    const float y_other = __shfl_xor_sync(0x0000ffffu, y, 1);   // lanes 2r, 2r+1 hold the two action components of row r
    if (row < a.n) {
      if (!a.a_out) a.y[row * 2 + j] = y;
      else if (j == 0) {
        const bool have = a.noise != nullptr;
        const ActOut o = act_gauss_epilogue(y, y_other, have, have ? a.noise[row] : 0.0f, have ? a.noise[a.ask + row] : 0.0f, a.sigma, a.seed,
                                            a.step, a.env_id_base + row, a.lo0, a.lo1, a.hi0, a.hi1);
        a.a_out[row] = o.a0; a.a_out[a.ask + row] = o.a1;
        if (a.scaled_out) { a.scaled_out[row] = o.s0; a.scaled_out[a.ask + row] = o.s1; }
        if (a.noise_acc) a.noise_acc[row] = __fadd_rn(a.noise_first ? 0.0f : a.noise_acc[row], o.noise_mean);
      }
    }
  }
}

int ddpg_fused_prepare() {
  CUDA_TRY(cudaFuncSetAttribute(ddpg_fused_critic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FusedSmem)));
  CUDA_TRY(cudaFuncSetAttribute(ddpg_fused_critic_nstep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FusedSmem)));
  CUDA_TRY(cudaFuncSetAttribute(ddpg_fused_actor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FusedSmem)));
  CUDA_TRY(cudaFuncSetAttribute(ddpg_fused_act_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FusedSmem)));
  return SHEMS_OK;
}
// launch as a programmatic dependent of the predecessor in the stream (captured as such in the update's graph)
template <typename K>
static int launch_pdl(K kernel, cudaStream_t st, const FusedArgs& a) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)((a.B / FUSED_ROWS) * FUSED_CLUSTER));
  cfg.blockDim = dim3(FT);
  cfg.dynamicSmemBytes = sizeof(FusedSmem);
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  CUDA_TRY(cudaLaunchKernelEx(&cfg, kernel, a));
  return SHEMS_OK;
}
// the critic pass opens the update (it reads what the previous update's optimiser wrote: an ordinary dependency) ...
int ddpg_fused_critic(cudaStream_t st, const FusedArgs& a) {
  if (a.links) ddpg_fused_critic_nstep_kernel<<<(a.B / FUSED_ROWS) * FUSED_CLUSTER, FT, sizeof(FusedSmem), st>>>(a);
  else ddpg_fused_critic_kernel<<<(a.B / FUSED_ROWS) * FUSED_CLUSTER, FT, sizeof(FusedSmem), st>>>(a);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}
// ... the actor pass is a programmatic dependent of ADAM(critic)
int ddpg_fused_actor(cudaStream_t st, const FusedArgs& a) { return launch_pdl(ddpg_fused_actor_kernel, st, a); }
int ddpg_fused_act(cudaStream_t st, const FusedActArgs& a) {
  const unsigned clusters = (unsigned)((a.n + FUSED_ROWS - 1) / FUSED_ROWS);
  ddpg_fused_act_kernel<<<clusters * FUSED_CLUSTER, FT, sizeof(FusedSmem), st>>>(a);
  CUDA_TRY(cudaGetLastError());
  return SHEMS_OK;
}
