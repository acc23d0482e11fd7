/*
 * oracle_weighted.c — test infrastructure: the CPU oracle's replay() body (oracle/ddpg_oracle.c) with importance weights on the
 * critic's output gradient, for the prioritized-replay tests.  It includes the oracle's source unchanged, so every helper (dense layers,
 * ADAM, soft_update!) is the oracle's own, and is built with the oracle's flags by tests/oracle_weighted.py into a temporary directory.
 */
#include "../oracle/ddpg_oracle.c"

/* oracle_ddpg_update_batch with importance weights w [B] (prioritized replay): the critic's output gradient of row b is
 * RN32(dq_b * w_b), everything else (the reported loss included) as there.  q_out, y_out [B] (or NULL) receive critic(s, a) and the
 * TD target of the critic step, from which the row's priority follows. */
void oracle_ddpg_update_batch_weighted(OracleDdpg* h, const float* s, const float* a, const float* r, const float* s2, const float* done,
                                       const float* w, float* q_out, float* y_out) {
  const int S = h->p.state_size, A = h->p.action_size, l1 = h->p.l1, l2 = h->p.l2, B = h->p.batch, C = S + A;
  float* xs = (float*)calloc((size_t)B * C, sizeof(float));   /* vcat(normalize(s), a)  */
  float* xs2 = (float*)calloc((size_t)B * C, sizeof(float));  /* vcat(normalize(s'), a') */
  float* sn = (float*)calloc((size_t)B * S, sizeof(float));
  float* s2n = (float*)calloc((size_t)B * S, sizeof(float));
  float* h1 = (float*)calloc((size_t)B * l1, sizeof(float)); float* h2 = (float*)calloc((size_t)B * l2, sizeof(float));
  float* g1 = (float*)calloc((size_t)B * l1, sizeof(float)); float* g2 = (float*)calloc((size_t)B * l2, sizeof(float));
  float* ah1 = (float*)calloc((size_t)B * l1, sizeof(float)); float* ah2 = (float*)calloc((size_t)B * l2, sizeof(float));
  float* a2 = (float*)calloc((size_t)B * A, sizeof(float)); float* api = (float*)calloc((size_t)B * A, sizeof(float));
  float* q = (float*)calloc((size_t)B, sizeof(float)); float* q2 = (float*)calloc((size_t)B, sizeof(float));
  float* y = (float*)calloc((size_t)B, sizeof(float)); float* dq = (float*)calloc((size_t)B, sizeof(float));
  float* dx = (float*)calloc((size_t)B * C, sizeof(float)); float* da = (float*)calloc((size_t)B * A, sizeof(float));

  normalize_into(h, s, B, sn, S); normalize_into(h, s2, B, s2n, S);
  /* a' = actor_target(normalize(s')); q' = critic_target(vcat(normalize(s'), a'))   :131-132 */
  net_fwd(&h->net[DDPG_NET_ACTOR_TARGET], s2n, B, h1, h2, a2);
  for (int b = 0; b < B; ++b) {
    for (int k = 0; k < S; ++k) { xs2[(size_t)b * C + k] = s2n[(size_t)b * S + k]; xs[(size_t)b * C + k] = sn[(size_t)b * S + k]; }
    for (int k = 0; k < A; ++k) { xs2[(size_t)b * C + S + k] = a2[(size_t)b * A + k]; xs[(size_t)b * C + S + k] = a[(size_t)k * B + b]; }
  }
  net_fwd(&h->net[DDPG_NET_CRITIC_TARGET], xs2, B, h1, h2, q2);
  /* y = r .+ γ .* (1 .- done) .* q'   :133 (Float32) */
  for (int b = 0; b < B; ++b) {
    const float nd = 1.f - (done ? done[b] : 0.f);
    const float t = h->p.gamma * nd;
    const float u = t * q2[b];
    y[b] = r[b] + u;
  }
  /* critic step :137, :114: loss = mean((critic(vcat(s_n, a)) - y)^2) */
  net_fwd(&h->net[DDPG_NET_CRITIC], xs, B, h1, h2, q);
  {
    double acc = 0.0;
    for (int b = 0; b < B; ++b) { const float d = q[b] - y[b]; acc += (double)(d * d); dq[b] = 2.f * d / (float)B; }
    h->loss_crit = (float)(acc / B);
    for (int b = 0; b < B; ++b) {
      dq[b] = dq[b] * w[b];
      if (q_out) q_out[b] = q[b];
      if (y_out) y_out[b] = y[b];
    }
  }
  {
    const Net* n = &h->net[DDPG_NET_CRITIC];
    dense_bwd(&n->l[2], h2, q, dq, B, h->gW[1][2], h->gb[1][2], g2);
    dense_bwd(&n->l[1], h1, h2, g2, B, h->gW[1][1], h->gb[1][1], g1);
    dense_bwd(&n->l[0], xs, h1, g1, B, h->gW[1][0], h->gb[1][0], NULL);
  }
  adam_net(h, DDPG_NET_CRITIC, h->p.lr_critic);
  /* actor step :140, :116-119: loss = -mean(critic(vcat(s_n, actor(s_n)))) with the UPDATED critic */
  net_fwd(&h->net[DDPG_NET_ACTOR], sn, B, ah1, ah2, api);
  for (int b = 0; b < B; ++b) for (int k = 0; k < A; ++k) xs[(size_t)b * C + S + k] = api[(size_t)b * A + k];
  net_fwd(&h->net[DDPG_NET_CRITIC], xs, B, h1, h2, q);
  {
    double acc = 0.0;
    for (int b = 0; b < B; ++b) { acc += (double)q[b]; dq[b] = -1.f / (float)B; }
    h->loss_act = (float)(-acc / B);
  }
  {
    const Net* c = &h->net[DDPG_NET_CRITIC];
    dense_bwd(&c->l[2], h2, q, dq, B, NULL, NULL, g2);
    dense_bwd(&c->l[1], h1, h2, g2, B, NULL, NULL, g1);
    dense_bwd(&c->l[0], xs, h1, g1, B, NULL, NULL, dx);
    for (int b = 0; b < B; ++b) for (int k = 0; k < A; ++k) da[(size_t)b * A + k] = dx[(size_t)b * C + S + k];
    const Net* n = &h->net[DDPG_NET_ACTOR];
    dense_bwd(&n->l[2], ah2, api, da, B, h->gW[0][2], h->gb[0][2], g2);
    dense_bwd(&n->l[1], ah1, ah2, g2, B, h->gW[0][1], h->gb[0][1], g1);
    dense_bwd(&n->l[0], sn, ah1, g1, B, h->gW[0][0], h->gb[0][0], NULL);
  }
  adam_net(h, DDPG_NET_ACTOR, h->p.lr_actor);
  /* :142-143 */
  soft_update(&h->net[DDPG_NET_ACTOR_TARGET], &h->net[DDPG_NET_ACTOR], h->p.tau);
  soft_update(&h->net[DDPG_NET_CRITIC_TARGET], &h->net[DDPG_NET_CRITIC], h->p.tau);

  free(xs); free(xs2); free(sn); free(s2n); free(h1); free(h2); free(g1); free(g2); free(ah1); free(ah2);
  free(a2); free(api); free(q); free(q2); free(y); free(dq); free(dx); free(da);
}
