"""Proportional prioritized replay on the device against its numpy restatement (tests/per_numpy.py) and the CPU oracle: the sum
tree's draws and weights bit for bit, the refresh of newly written slots, α = 0 as exact uniform weighting, the weighted critic step
and the priority write-back, resume, populations and the calls a prioritized handle refuses."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import oracle_weighted as OW  # noqa: E402
import per_numpy as PN  # noqa: E402

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def dev(x):
    return torch.as_tensor(np.ascontiguousarray(x), device="cuda")


def push_random(mem, rng, n):
    s, s2 = rng.uniform(-1, 3, (9, n)).astype(np.float32), rng.uniform(-1, 3, (9, n)).astype(np.float32)
    a, r = rng.uniform(-1, 1, (2, n)).astype(np.float32), rng.uniform(-5, 1, n).astype(np.float32)
    mem.push(dev(s), dev(a), dev(r), dev(s2))


def leaves_by_slot(mem):
    """the memory's priorities by physical slot (unfilled slots 0)"""
    prio, _ = mem.priorities()
    cap, head, n = mem.capacity, mem.head, len(mem)
    out = np.zeros(cap, np.float32)
    out[(head - n + np.arange(n)) % cap] = prio
    return out


def check_sample(O, mem, seed, B, beta):
    idx, w = mem.sample_prioritized(B, seed=seed, beta=beta)
    idx, w = idx.cpu().numpy(), w.cpu().numpy()
    leaves = leaves_by_slot(mem)
    want_idx, want_w, slots = PN.sample(O, leaves, mem.capacity, mem.head, len(mem), seed, B, beta)
    np.testing.assert_array_equal(idx, want_idx)
    np.testing.assert_array_equal(w.view(np.uint32), want_w.view(np.uint32))
    prio, _ = mem.priorities()
    assert np.all(prio[idx] > 0), "a draw landed on a zero-priority slot"
    return idx, w


@pytest.mark.parametrize("cap,pushes", [(1000, [700]), (37, [20, 30, 25]), (4096, [5000]), (3, [1])])
def test_sampling_matches_restatement(sb, O, cap, pushes):
    rng = np.random.default_rng(cap)
    mem = sb.Replay(cap)
    push_random(mem, rng, pushes[0])
    mem.enable_priorities()
    prio, pmax = mem.priorities()
    assert pmax == 1.0 and np.all(prio == 1.0)
    for n in pushes[1:]:
        push_random(mem, rng, n)
    for seed, B, beta in [(1, 120, 0.4), (77, 33, 1.0), (5, 512, 0.0)]:
        check_sample(O, mem, seed, B, beta)
    # priorities with zeros and values whose Float32 sums round
    n = len(mem)
    p = rng.choice(np.array([0.0, 1e-7, 3.0, 1e7, 0.3, 1.0 + 2**-23], np.float32), n)
    p[rng.integers(0, n)] = 2.5
    mem.set_priorities(p, 1e7)
    got, pm = mem.priorities()
    np.testing.assert_array_equal(got, p)
    assert pm == np.float32(1e7)
    for seed, B, beta in [(2, 120, 0.4), (9, 257, 0.7)]:
        check_sample(O, mem, seed, B, beta)
    with pytest.raises(sb.ShemsError):
        mem.set_priorities(np.zeros(n, np.float32), 1.0)
    with pytest.raises(sb.ShemsError):
        mem.set_priorities(np.full(n, -1.0, np.float32), 1.0)


def test_sampling_compact_records(sb, O, train_series):
    n, T = 256, 40
    env = sb.Shems(T, train_series, n_envs=n)
    mem = sb.Replay(n * T)
    env.reset(rng=3)
    env.rollout(sb.POLICY_RANDOM, T, seed=3, replay=mem, want_return=False)
    assert mem.series_copies == 1
    mem.enable_priorities()
    rng = np.random.default_rng(1)
    mem.set_priorities(rng.uniform(0, 4, len(mem)).astype(np.float32), 4.0)
    idx, _ = check_sample(O, mem, 11, 120, 0.5)
    S, A, R, S2, D = mem.get()
    s, a, r, s2, d = mem.sample(120, idx=idx)
    np.testing.assert_array_equal(s.cpu().numpy(), S[:, idx])
    np.testing.assert_array_equal(r.cpu().numpy(), R[idx])


def test_refresh_after_writers(sb, train_series):
    rng = np.random.default_rng(5)
    mem = sb.Replay(100)
    push_random(mem, rng, 60)
    mem.enable_priorities()
    mem.set_priorities(rng.uniform(0.1, 2, 60).astype(np.float32), 7.0)
    before, _ = mem.priorities()
    push_random(mem, rng, 30)                     # replay_push
    after, pm = mem.priorities()
    np.testing.assert_array_equal(after[:60], before)
    assert pm == 7.0 and np.all(after[60:] == 7.0)
    mem.set_priorities(after * np.float32(0.5), 3.0)
    push_random(mem, rng, 250)                    # n > cap: every slot is new
    after, _ = mem.priorities()
    assert len(after) == 100 and np.all(after == 3.0)
    # replay_push_groups
    mems = [sb.Replay(50), sb.Replay(80)]
    for m in mems:
        push_random(m, rng, 40)
        m.enable_priorities()
        m.set_priorities(rng.uniform(0.1, 2, 40).astype(np.float32), 5.0)
    old = [m.priorities()[0] for m in mems]
    N = 2 * 25
    s = dev(rng.normal(size=(9, N)).astype(np.float32))
    sb.ddpg.push_groups(mems, s, dev(rng.normal(size=(2, N)).astype(np.float32)), dev(rng.normal(size=N).astype(np.float32)), s)
    for m, o in zip(mems, old):
        p, _ = m.priorities()
        keep = len(p) - 25
        np.testing.assert_array_equal(p[:keep], o[len(o) - keep:])
        assert np.all(p[keep:] == 5.0)
    # a rollout with a replay sink (wrapping)
    n, T = 64, 10
    env = sb.Shems(T, train_series, n_envs=n)
    mem = sb.Replay(n * 16)
    env.reset(rng=1)
    env.rollout(sb.POLICY_RANDOM, T, seed=1, replay=mem, want_return=False)
    mem.enable_priorities()
    mem.set_priorities(rng.uniform(0.1, 2, len(mem)).astype(np.float32), 9.0)
    old, _ = mem.priorities()
    env.reset(rng=2)
    env.rollout(sb.POLICY_RANDOM, T, seed=2, replay=mem, want_return=False)
    p, _ = mem.priorities()
    keep = len(p) - n * T
    np.testing.assert_array_equal(p[:keep], old[len(old) - keep:])
    assert np.all(p[keep:] == 9.0)
    # ddpg_episode (no update: the written slots alone change)
    le = sb.Learner()
    le.init(1)
    le.set_prioritized(0.6, 0.4)
    env.reset(rng=3)
    old, _ = mem.priorities()
    le.episode(env, mem, 5, train=True, rng_ep=3, updates_per_step=0)
    p, _ = mem.priorities()
    keep = len(p) - n * 5
    np.testing.assert_array_equal(p[:keep], old[len(old) - keep:])
    assert np.all(p[keep:] == 9.0)


def _pair(sb, P=1, **kw):
    per = sb.Learner(params=sb.default_ddpg_params(population=P, **kw))
    plain = sb.Learner(params=sb.default_ddpg_params(population=P, **kw))
    per.init(21)
    plain.init(21)
    plain.set_fused(False)
    return per, plain


@pytest.mark.parametrize("B,tc,P,cap", [(120, 0, 1, 3000), (8192, 1, 1, 20000), (120, 0, 4, 1500)])
def test_alpha0_is_uniform_weighting(sb, O, B, tc, P, cap):
    rng = np.random.default_rng(B + P)
    per, plain = _pair(sb, P, batch=B, use_tensor_cores=tc)
    mems = []
    for _ in range(P):
        m = sb.Replay(cap)
        push_random(m, rng, cap - 7)
        m.enable_priorities()
        mems.append(m)
    K, seed = 3, 41
    per.set_prioritized(0.0, 0.7, 1e-3)
    idx = np.zeros((P, K, B), np.int32)
    for l, m in enumerate(mems):
        t, p2 = PN.build_tree(leaves_by_slot(m), cap)
        for u in range(K):
            slots = [PN.draw(O, t, p2, seed + l, j, u, B)[0] for j in range(B)]
            idx[l, u] = [PN.logical(s, m.head, len(m), cap) for s in slots]
    if P == 1:
        per.replay(mems[0], rng_rpl=seed, n_updates=K)
        plain.replay(mems[0], n_updates=K, idx=idx[0])
    else:
        per.replay(mems, rng_rpl=seed, n_updates=K)
        plain.replay(mems, n_updates=K, idx=idx)
    for l in range(P):
        per.select(l)
        plain.select(l)
        for net in range(4):
            for k in range(3):
                for x, y in zip(per.get_layer(net, k), plain.get_layer(net, k)):
                    np.testing.assert_array_equal(x.view(np.uint32), y.view(np.uint32))
        p, pm = mems[l].priorities()
        assert pm == 1.0 and np.all(p == 1.0)


@pytest.mark.parametrize("B,l1,l2,tc,K", [(120, 250, 500, 0, 3), (1024, 250, 500, 1, 2)])
def test_weighted_update_vs_oracle(sb, O, B, l1, l2, tc, K, tmp_path):
    WL = OW.load(str(tmp_path))
    rng = np.random.default_rng(B)
    kw = dict(batch=B, l1=l1, l2=l2)
    orc = O.OracleDdpg(O.default_ddpg_params(**kw))
    orc.init(5)
    le = sb.Learner(params=sb.default_ddpg_params(use_tensor_cores=tc, **kw))
    for net in range(4):
        for k in range(3):
            le.set_layer(net, k, *orc.get_layer(net, k))
    s_min = rng.uniform(-1, 0, 9).astype(np.float32)
    s_max = (s_min + rng.uniform(0.5, 3, 9)).astype(np.float32)
    orc.set_norm(s_min, s_max)
    le.set_norm(s_min, s_max)
    cap = 3 * B
    mem = sb.Replay(cap)
    push_random(mem, rng, cap + B // 2)            # wrapped
    mem.enable_priorities()
    mem.set_priorities(rng.uniform(0.05, 3.0, cap).astype(np.float32), 3.0)
    alpha, beta, eps = 0.6, 0.4, 1e-3
    le.set_prioritized(alpha, beta, eps)
    S, A, R, S2, D = mem.get()
    g_rtol, g_atol, l_rel = (2e-4, 2e-6, 1e-4) if not tc else (0.0, 1e-2, 2e-3)
    for step in range(K):
        idx = rng.integers(0, cap, B).astype(np.int32)
        idx[1] = idx[0]                             # a slot drawn twice
        prio, pmax = mem.priorities()
        t, _ = PN.build_tree(leaves_by_slot(mem), cap)
        w = PN.weights(prio[idx], cap, t[1], beta)
        q, y = OW.update_batch_weighted(WL, orc, S[:, idx], A[:, idx], R[idx], S2[:, idx], D[idx], w)
        le.replay(mem, idx=idx)
        if step == 0:
            for net in (0, 1):
                for k in range(3):
                    gw, gb = le.get_grad(net, k)
                    ow, ob = orc.get_grad(net, k)
                    sc = max(np.abs(ow).max(), 1e-12)
                    np.testing.assert_allclose(gw, ow, rtol=g_rtol, atol=g_atol * sc)
                    np.testing.assert_allclose(gb, ob, rtol=g_rtol, atol=g_atol * max(np.abs(ob).max(), 1e-12))
        lc, la = le.losses()
        olc, ola = orc.losses()
        assert lc == pytest.approx(olc, rel=l_rel) and la == pytest.approx(ola, rel=l_rel, abs=1e-6)
        # write-back: the largest p_j of the rows that drew a slot; the rest unchanged; p_max
        new, new_pmax = mem.priorities()
        want = {}
        for j, i in enumerate(idx):
            want[i] = max(want.get(i, 0.0), float(PN.priority(y[j], q[j], alpha, eps)))
        rows = np.array(sorted(want))
        np.testing.assert_allclose(new[rows], [want[i] for i in rows], rtol=1e-3 if not tc else 2e-2, atol=1e-5)
        untouched = np.setdiff1d(np.arange(cap), rows)
        np.testing.assert_array_equal(new[untouched], prio[untouched])
        assert new_pmax == max(pmax, new[rows].max())


def test_resume_is_bit_identical(sb, train_series, tmp_path):
    n, T = 64, 24
    env = sb.Shems(T, train_series, n_envs=n)

    def setup():
        le = sb.Learner()
        le.init(3)
        mem = sb.Replay(3000)                       # wraps in the second episode
        le.set_prioritized(0.6, 0.5, 1e-4)
        return le, mem

    def run(le, mem, episodes):
        for e in episodes:
            env.reset(rng=100 + e)
            le.episode(env, mem, T, train=True, rng_ep=e, updates_per_step=1)

    le, mem = setup()
    env.reset(rng=99)
    env.rollout(sb.POLICY_RANDOM, T, seed=99, replay=mem, want_return=False)
    mem.enable_priorities()
    le.set_norm(*mem.min_max_buffer(len(mem), rng_mm=1))
    run(le, mem, [1, 2])
    path = str(tmp_path / "ck.npz")
    sb.tracker.save_checkpoint(path, le, memories=mem)
    head = mem.head
    assert len(mem) == mem.capacity and head != 0   # a full, wrapped memory: the restore must rebuild the slot order
    run(le, mem, [3, 4])
    le2, mem2 = setup()
    sb.tracker.load_checkpoint(path, le2, memories=mem2)
    assert mem2.head == head
    run(le2, mem2, [3, 4])
    for net in range(4):
        for k in range(3):
            for x, y in zip(le.get_layer(net, k), le2.get_layer(net, k)):
                np.testing.assert_array_equal(x.view(np.uint32), y.view(np.uint32))
    np.testing.assert_array_equal(mem.priorities()[0], mem2.priorities()[0])
    assert mem.priorities()[1] == mem2.priorities()[1]


def test_population_equals_single_learners(sb):
    P, B, K, cap = 3, 120, 4, 2000
    rng = np.random.default_rng(8)
    pop = sb.Learner(params=sb.default_ddpg_params(population=P, batch=B))
    pop.init(50)
    pop.set_prioritized(0.6, 0.4, 1e-3)
    pm, singles, sm = [], [], []
    for l in range(P):
        a, b = sb.Replay(cap), sb.Replay(cap)
        st = np.random.default_rng(100 + l)
        push_random(a, st, cap)
        push_random(b, np.random.default_rng(100 + l), cap)
        a.enable_priorities()
        b.enable_priorities()
        pm.append(a)
        sm.append(b)
        le = sb.Learner(params=sb.default_ddpg_params(batch=B))
        le.init(50 + l)
        le.set_prioritized(0.6, 0.4, 1e-3)
        singles.append(le)
    pop.replay(pm, rng_rpl=7, n_updates=K)
    for l, le in enumerate(singles):
        le.replay(sm[l], rng_rpl=7 + l, n_updates=K)
        pop.select(l)
        for net in range(4):
            lr = pop.p.lr_actor if net in (0, 2) else pop.p.lr_critic
            for k in range(3):
                for x, y in zip(pop.get_layer(net, k), le.get_layer(net, k)):
                    np.testing.assert_allclose(x, y, rtol=1e-5, atol=0.02 * lr * K + 1e-7)
        np.testing.assert_allclose(pm[l].priorities()[0], sm[l].priorities()[0], rtol=1e-3, atol=1e-5)


def test_rejections(sb, train_series):
    rng = np.random.default_rng(2)
    le = sb.Learner()
    le.init(4)
    plain_mem, mem = sb.Replay(500), sb.Replay(500)
    push_random(plain_mem, rng, 300)
    push_random(mem, rng, 300)
    mem.enable_priorities()
    for bad in [(-0.1, 0.4, 1e-6), (0.6, 1.5, 1e-6), (0.6, 0.4, 0.0), (float("nan"), 0.4, 1e-6), (0.6, float("inf"), 1e-6)]:
        with pytest.raises(sb.ShemsError):
            le.set_prioritized(*bad)
    assert le.get_prioritized() is None
    obs = dev(rng.uniform(0, 1, (9, 16)).astype(np.float32))
    a0, _ = le.act(obs, train=False)
    le.set_prioritized(0.6, 0.4, 1e-6)
    assert le.get_prioritized()["alpha"] == np.float32(0.6)
    before = [le.get_layer(n, k)[0].copy() for n in range(4) for k in range(3)]
    with pytest.raises(sb.ShemsError):
        le.replay(plain_mem, rng_rpl=1)             # memory without priorities
    s = dev(rng.normal(size=(9, 120)).astype(np.float32))
    with pytest.raises(sb.ShemsError):
        le.update_batch(s, dev(np.zeros((2, 120), np.float32)), dev(np.zeros(120, np.float32)), s)
    with pytest.raises(sb.ShemsError):
        le.replay_dp(mem)                           # ddpg_update_phase
    with pytest.raises(sb.ShemsError):
        le.replay_fused_dp(mem)                     # ddpg_update_dp
    with pytest.raises(sb.ShemsError):
        le.dp_connect(0, 1, [le.dp_export()])
    env = sb.Shems(8, train_series, n_envs=32)
    env.reset(rng=1)
    with pytest.raises(sb.ShemsError):
        le.episode(env, plain_mem, 4, train=True)
    after = [le.get_layer(n, k)[0] for n in range(4) for k in range(3)]
    for x, y in zip(before, after):
        np.testing.assert_array_equal(x, y)
    prio, _ = mem.priorities()
    assert np.all(prio == 1.0)
    a1, _ = le.act(obs, train=False)                # act() keeps its path and bits
    np.testing.assert_array_equal(a0.cpu().numpy(), a1.cpu().numpy())
    pop = sb.Learner(params=sb.default_ddpg_params(population=2))
    pop.set_prioritized(0.6, 0.4, 1e-6)
    with pytest.raises(sb.ShemsError):
        pop.replay([mem, mem], rng_rpl=1)           # two prioritized learners cannot share a memory
