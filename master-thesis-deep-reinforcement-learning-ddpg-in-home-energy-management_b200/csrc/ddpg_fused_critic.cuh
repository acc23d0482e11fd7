// ddpg_fused_critic.cuh — the critic pass of the cluster-fused update, included twice by ddpg_fused.cu: as ddpg_fused_critic_kernel
// (FUSED_CRITIC_NSTEP 0) and as ddpg_fused_critic_nstep_kernel (FUSED_CRITIC_NSTEP 1).  The n-step kernel's prologue walks each row's
// chain from the drawn record (ring.cuh ring_nstep over a.links[0], n = *a.nstep, the learner's γ) and takes s', r and done from the
// walk, so the unchanged TD target below is the n-step target.  (One source compiled twice rather than a template: the 1-step kernel
// keeps its instruction stream exactly.)
// No include guard: FUSED_CRITIC_KERNEL and FUSED_CRITIC_NSTEP are defined by the includer.
__global__ void __cluster_dims__(FUSED_CLUSTER, 1, 1) __launch_bounds__(FT, 1)
FUSED_CRITIC_KERNEL(const FusedArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FusedSmem* S = reinterpret_cast<FusedSmem*>(smem_raw);
  cg::cluster_group cluster = cg::this_cluster();
  const int tid = threadIdx.x, lane = tid & 31;
  const Geo g = make_geo(a.l1, a.l2, a.vec16, cluster);
  const int l1 = a.l1, l2 = a.l2;
  float* part = a.part + (long long)(blockIdx.x / FUSED_CLUSTER) * a.part_stride;
  const bool vec16 = a.vec16 != 0;   // 16-byte aligned W2 rows: vector staging and vector shared-memory reads
STAMP(0, 0);
    cluster_arrive();  // "this CTA runs": waited for before the first write into a peer's shared memory
  STAMP(0, 16);
  // the cluster's 8 transitions: ring_draw (or host-supplied) indices into the replay ring, as ddpg_gather_kernel draws them, or the
  // rows of a caller-supplied minibatch
  const float* ring = a.rings ? a.rings[0] : nullptr;
  if (tid < 8) {
    const int j = g.row0 + tid;
    unsigned long long where = (unsigned long long)j;
    const float* ser = nullptr;
    if (ring) {
      const long long len = a.ctrl->len, head = a.ctrl->head, cap = a.ctrl->cap;
      const long long li = a.ctrl->use_idx ? a.idx[(long long)a.ctrl->idx_cursor * a.B + j] : ring_draw(a.ctrl->seed, j, a.ctrl->update, len);
      where = (unsigned long long)ring_base(ring_slot(li, head, len, cap));
      ser = ring_row(ring_table(ring), ring + where);
#if FUSED_CRITIC_NSTEP
      {
        const RingNstep w = ring_nstep(ring, ring_table(ring), a.links[0], ring_slot(li, head, len, cap), *a.nstep, a.ctrl->hp.gamma, true);
        S->ns_row[tid] = (unsigned long long)ring_base(w.last);
        S->ns_ser[tid] = ring_row(ring_table(ring), ring + ring_base(w.last));
        S->ns_r[tid] = w.r;
        S->ns_d[tid] = w.done;
      }
#endif
    }
    S->src_row[tid] = where;
    S->src_ser[tid] = ser;
  }
  stage_w2(S->W[0], a.actor_t + a.ao.w2, l1, l2, g.n0, g.nv, vec16, tid);   // slot 0: actor_target W2
  STAMP(0, 17);
  stage_w2(S->W[1], a.critic + a.co.w2, l1, l2, g.n0, g.nv, vec16, tid);    // slot 1: critic W2
  STAMP(0, 18);
  // the small operands of all three nets, into registers: one exposed global-memory latency for the whole kernel
  const L1Regs Rat = load_l1(a.actor_t + a.ao.w1, a.actor_t + a.ao.b1, 9, l1, tid);
  const L1Regs Rc = load_l1(a.critic + a.co.w1, a.critic + a.co.b1, 11, l1, tid);
  const L1Regs Rct = load_l1(a.critic_t + a.co.w1, a.critic_t + a.co.b1, 11, l1, tid);
  const TailRegs Tat = load_tail(a.actor_t + a.ao.b2 + g.n0, a.actor_t + a.ao.w3 + g.n0 * 2, 2, g.nv, lane);
  const TailRegs Tc = load_tail(a.critic + a.co.b2 + g.n0, a.critic + a.co.w3 + g.n0, 1, g.nv, lane);
  const TailRegs Tct = load_tail(a.critic_t + a.co.b2 + g.n0, a.critic_t + a.co.w3 + g.n0, 1, g.nv, lane);
  const float w3c = ((tid & 63) < g.nv) ? __ldg(a.critic + a.co.w3 + g.n0 + (tid & 63)) : 0.0f;   // b3: column tid & 63
  const float b3at = __ldg(a.actor_t + a.ao.b3 + (tid & 1)), b3c = __ldg(a.critic + a.co.b3), b3ct = __ldg(a.critic_t + a.co.b3);
  STAMP(0, 19);
  __syncthreads();   // src_row
  if (tid < 8 * RING_TRANSITION_FIELDS) {  // thread = (row, field): the ring's field order s[9] a[2] r s'[9] done
    const int r = tid / RING_TRANSITION_FIELDS, f = tid - r * RING_TRANSITION_FIELDS;
    const unsigned long long where = S->src_row[r];
    float v;
#if FUSED_CRITIC_NSTEP
    if (f >= RING_R) v = f == RING_R ? S->ns_r[r] : f == RING_DONE ? S->ns_d[r] : ring_field(ring + S->ns_row[r], S->ns_ser[r], f);
    else
#endif
    if (ring) v = ring_field(ring + where, S->src_ser[r], f);
    else if (f < RING_A) v = a.src_s[(long long)f * a.src_ld + where];
    else if (f < RING_R) v = a.src_a[(long long)(f - RING_A) * a.src_ld + where];
    else if (f == RING_R) v = a.src_r[where];
    else if (f < RING_DONE) v = a.src_s2[(long long)(f - RING_S2) * a.src_ld + where];
    else v = a.src_d ? a.src_d[where] : 0.0f;
    const bool is_s = f < RING_A, is_s2 = f >= RING_S2 && f < RING_DONE;
    if (is_s || is_s2) {  // normalize(s) = (s - s_min) / (s_max - s_min + 1f-8)
      const int k = is_s ? f : f - RING_S2;
      const float lo = a.norm[k];
      const float den = __fadd_rn(__fsub_rn(a.norm[9 + k], lo), 1e-8f);
      v = __fdiv_rn(__fsub_rn(v, lo), den);
      if (is_s) S->x[1][r * 12 + k] = v; else S->x[0][r * 12 + k] = v;       // (s_n | a) and s'_n
    } else if (f < RING_R) S->x[1][r * 12 + f] = v;
    else if (f == RING_R) S->rr[r] = v;
    else S->dd[r] = v;
  }
  STAMP(0, 20);
  __syncthreads();   // x
  STAMP(0, 1);
  // actor_target(s'_n)
  f1(Rat, 9, l1, S->x[0], S->h1T[0], tid);
  cp_wait<1>();
  __syncthreads();
  STAMP(0, 2);
  f2(S->W[0], Tat, l1, g.nv, S->h1T[0], S->red, S->h2s[0], tid);
  STAMP(0, 3);
  stage_w2(S->W[0], a.critic_t + a.co.w2, l1, l2, g.n0, g.nv, vec16, tid);  // slot 0 is free again: critic_target W2
  cluster_wait();    // every CTA of the cluster runs: its shared memory may be written from now on
  f3_partial(Tat, S->h2s[0], S, 0, cluster, g.rank, tid);
  STAMP(0, 4);
  // critic(s_n, a)
  f1(Rc, 11, l1, S->x[1], S->h1T[1], tid);
  cp_wait<1>();
  __syncthreads();
  STAMP(0, 5);
  f2(S->W[1], Tc, l1, g.nv, S->h1T[1], S->red, S->h2s[1], tid);
  STAMP(0, 6);
  f3_partial(Tc, S->h2s[1], S, 1, cluster, g.rank, tid);
  cluster.sync();
  STAMP(0, 7);
  if (tid < 16) {
    const int r = tid >> 1, j = tid & 1;
    S->x[0][r * 12 + 9 + j] = tanhf(xch_sum(S, 0, r, j) + b3at);   // a' -> vcat(s'_n, a')
  } else if (tid >= 32 && tid < 40) {
    const int r = tid - 32;
    S->qv[r] = xch_sum(S, 1, r, 0) + b3c;
  }
  __syncthreads();
  // critic_target(s'_n, a')
  f1(Rct, 11, l1, S->x[0], S->h1T[0], tid);
  cp_wait<0>();   // second use of slot 0
  __syncthreads();
  STAMP(0, 8);
  f2(S->W[0], Tct, l1, g.nv, S->h1T[0], S->red, S->h2s[0], tid);
  STAMP(0, 9);
  f3_partial(Tct, S->h2s[0], S, 2, cluster, g.rank, tid);
  cluster.sync();
  STAMP(0, 10);
  if (tid < 8) {  // y = r + γ(1-done) q'  (:133);  d mse / d q = 2 (q - y) / B
    const int r = tid;
    const float q2 = xch_sum(S, 2, r, 0) + b3ct;
    const float y = S->rr[r] + (a.ctrl->hp.gamma * (1.0f - S->dd[r])) * q2;
    S->dout[r * 2] = 2.0f * (S->qv[r] - y) * a.inv_batch;
    S->dout[r * 2 + 1] = 0.0f;
    S->rr[r] = y;
  }
  __syncthreads();
  // critic backward.  Everything that goes to global memory waits until after the last cluster barrier: the barrier's release
  // fence would otherwise sit on the outstanding stores.
  b3_dz(w3c, 0.0f, 1, g.nv, S->h2s[1], S->dout, S->dzT, tid);
  __syncthreads();
  STAMP(0, 11);
  bx2(S->W[1], S->dzT, l1, g.nv, g.n1s, vec16, S, cluster, g.rank, tid);
  STAMP(0, 12);
  cluster.sync();
  STAMP(0, 13);
  if (g.rank == 0) {
    if (tid < 8) { a.q[g.row0 + tid] = S->qv[tid]; a.y[g.row0 + tid] = S->rr[tid]; }
    else if (tid >= 32 && tid < 32 + 88) {  // the gathered (s_n | a) rows, for the actor pass
      const int e = tid - 32, r = e / 11, i = e - r * 11;
      a.xs_w[(long long)(g.row0 + r) * 11 + i] = S->x[1][r * 12 + i];
    }
  }
  b3_grads(1, g.nv, S->h2s[1], S->dout, part + a.co.w3 + g.n0, g.rank == 0 ? part + a.co.b3 : nullptr, tid);
  bw2(S->h1T[1], S->dzT, l1, l2, g.nv, part + a.co.w2 + g.n0, part + a.co.b2 + g.n0, tid);
  STAMP(0, 14);
  rs_finish(S, S->h1T[1], g.k0, g.n1v, tid);
  __syncthreads();
  bw1(S->x[1], 11, S->dz1s, l1, g.n1v, part + a.co.w1 + g.k0, part + a.co.b1 + g.k0, tid);
  STAMP(0, 15);
}
