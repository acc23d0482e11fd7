"""n-step returns on the device against their numpy restatement (tests/nstep_numpy.py), bit for bit: the successor links after every
writer, replay_sample_nstep, every update regime against a "materialised twin" (a 1-step learner with the same weights trained on the
n-step minibatch pushed into a fresh memory), prioritized n-step updates, n = 1, resume, and the calls an n-step handle refuses."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import nstep_numpy as NN  # noqa: E402

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def dev(x):
    return torch.as_tensor(np.ascontiguousarray(x), device="cuda")


def check_write(mem, write, n_written, width):
    """run one write and compare the device's links with the rule applied to the links before it"""
    prev, n0 = mem.successors(), len(mem)
    write()
    S, A, R, S2, D = mem.get()
    want = NN.after_write(prev, n0, S, S2, D, n_written, width, mem.capacity)
    got = mem.successors()
    np.testing.assert_array_equal(got, want)
    return got


def check_steps(mem, write, steps, width):
    """a call that makes `steps` writes of `width` records each without wrapping (ddpg_episode): the rule write by write"""
    nx, n0 = mem.successors(), len(mem)
    write()
    S, A, R, S2, D = mem.get()
    assert len(mem) == n0 + steps * width, "keep the memory from wrapping here"
    for t in range(steps):
        e = n0 + (t + 1) * width
        nx = NN.after_write(nx, e - width, S[:, :e], S2[:, :e], D[:e], width, width, mem.capacity)
    np.testing.assert_array_equal(mem.successors(), nx)
    return nx


class Walker:
    """n instances of random 9-dimensional states: step() -> (s, a, r, s', done) where some instances end (done = 1) or restart
    (their next s is a fresh state), the others continue from s'"""

    def __init__(self, rng, n):
        self.rng, self.n = rng, n
        self.s = rng.standard_normal((9, n)).astype(np.float32)

    def step(self):
        rng, n = self.rng, self.n
        s2 = rng.standard_normal((9, n)).astype(np.float32)
        done = (rng.uniform(size=n) < 0.1).astype(np.float32)
        out = (self.s, rng.uniform(-1, 1, (2, n)).astype(np.float32), rng.standard_normal(n).astype(np.float32), s2, done)
        self.s = np.where(rng.uniform(size=n) < 0.15, rng.standard_normal((9, n)).astype(np.float32), s2)
        return out


def test_links_after_every_writer(sb, train_series, monkeypatch):
    rng = np.random.default_rng(0)
    # replay_push, one step of 4 instances at a time, wrapping; a push of one record; a push larger than the memory
    mem = sb.Replay(100).enable_successors()
    w = Walker(rng, 4)
    for _ in range(40):
        s, a, r, s2, d = w.step()
        check_write(mem, lambda: mem.push(dev(s), dev(a), dev(r), dev(s2), dev(d)), 4, 4)
    s, a, r, s2, d = Walker(rng, 1).step()
    check_write(mem, lambda: mem.push(dev(s), dev(a), dev(r), dev(s2), dev(d)), 1, 1)
    w = Walker(rng, 150)
    s, a, r, s2, d = w.step()
    check_write(mem, lambda: mem.push(dev(s), dev(a), dev(r), dev(s2), dev(d)), 150, 150)
    assert (mem.successors() == -1).all()
    # replay_push_groups: 2 learners of 5 instances, the first memory wraps
    mems = [sb.Replay(50).enable_successors(), sb.Replay(80).enable_successors()]
    w = Walker(rng, 10)
    for _ in range(12):
        s, a, r, s2, d = w.step()
        prev = [(m.successors(), len(m)) for m in mems]
        sb.ddpg.push_groups(mems, dev(s), dev(a), dev(r), dev(s2), dev(d))
        for l, m in enumerate(mems):
            S, A, R, S2, D = m.get()
            np.testing.assert_array_equal(m.successors(), NN.after_write(prev[l][0], prev[l][1], S, S2, D, 5, 5, m.capacity))
    # rollouts: compact and full records, trimmed and general kernels; a memory that wraps and a rollout larger than the memory
    n, T = 64, 10
    env = sb.Shems(T, train_series, n_envs=n)
    for compact, lean in ((1, 1), (0, 1), (1, 0), (0, 0)):
        monkeypatch.setenv("SHEMS_RING_COMPACT", str(compact))
        monkeypatch.setenv("SHEMS_ROLLOUT_LEAN", str(lean))
        for cap in (n * 16, n * 4):
            mem = sb.Replay(cap).enable_successors()
            for ep in range(2):
                env.reset(rng=10 * compact + lean + ep)
                nx = check_write(mem, lambda: env.rollout(sb.POLICY_RANDOM, T, seed=ep, replay=mem, want_return=False), n * T, n)
            assert mem.series_copies == compact
            assert (nx >= 0).sum() > len(mem) // 2, "a rollout's steps are linked"
    monkeypatch.delenv("SHEMS_RING_COMPACT")
    monkeypatch.delenv("SHEMS_ROLLOUT_LEAN")
    # ddpg_episode: one learner (its post-step kernel) and a population (replay_push_groups), after a rollout into the same memory
    le = sb.Learner()
    le.init(1)
    le.set_nstep(3)
    mem = sb.Replay(n * 40).enable_successors()
    env.reset(rng=5)
    env.rollout(sb.POLICY_RANDOM, T, seed=5, replay=mem, want_return=False)
    env.reset(rng=6)
    check_steps(mem, lambda: le.episode(env, mem, 5, train=True, rng_ep=6, updates_per_step=0), 5, n)
    pop = sb.Learner(params=sb.default_ddpg_params(population=2))
    pop.init(2)
    pop.set_nstep(2)
    mems = [sb.Replay(400).enable_successors(), sb.Replay(400).enable_successors()]
    env.reset(rng=7)
    prev = [m.successors() for m in mems]
    pop.episode(env, mems, 6, train=True, rng_ep=7, updates_per_step=0)
    for m, nx in zip(mems, prev):
        S, A, R, S2, D = m.get()
        for t in range(6):
            e = (t + 1) * (n // 2)
            nx = NN.after_write(nx, e - n // 2, S[:, :e], S2[:, :e], D[:e], n // 2, n // 2, m.capacity)
        np.testing.assert_array_equal(m.successors(), nx)


def rollout_memory(sb, series, cap, n, T, episodes, seed):
    mem = sb.Replay(cap).enable_successors()
    env = sb.Shems(T, series, n_envs=n)
    for e in range(episodes):
        env.reset(rng=seed + e)
        env.rollout(sb.POLICY_RANDOM, T, seed=seed + e, replay=mem, want_return=False)
    return mem


def test_sample_nstep_matches_restatement(sb, O, train_series):
    mem = rollout_memory(sb, train_series, 4096, 128, 12, 2, 3)
    w = Walker(np.random.default_rng(4), 8)       # full records with terminal steps
    for _ in range(6):
        s, a, r, s2, d = w.step()
        mem.push(dev(s), dev(a), dev(r), dev(s2), dev(d))
    S, A, R, S2, D = mem.get()
    nx = mem.successors()
    # a link out of a terminal record (set_successors accepts it): the walk must still stop there
    term = np.flatnonzero(D == 1)
    assert term.size and term[0] + 1 < len(mem)
    nx[term[0]] = term[0] + 1
    mem.set_successors(nx)
    np.testing.assert_array_equal(mem.successors(), nx)
    B = 300
    for n in (2, 3, 8, 16):
        for gamma, seed in ((0.99, 11), (0.9, 12), (0.5, 13), (1.0, 14)):
            got = [x.cpu().numpy() for x in mem.sample_nstep(B, seed=seed, n=n, gamma=gamma)]
            idx = O.sample_indices(seed, 0, len(mem), B)
            want = NN.sample(S, A, R, S2, D, nx, idx, n, gamma)
            for g, x in zip(got, want):
                np.testing.assert_array_equal(g.view(np.uint32), x.view(np.uint32))
            assert got[5].max() == min(n, 12)      # the rollouts' episodes are 12 steps long
        t0 = term[:4]
        idx = np.concatenate([t0, O.sample_indices(99, 0, len(mem), 60)]).astype(np.int32)
        got = [x.cpu().numpy() for x in mem.sample_nstep(idx.size, n=n, gamma=0.97, idx=idx)]
        want = NN.sample(S, A, R, S2, D, nx, idx, n, 0.97)
        assert np.all(got[5][:t0.size] == 1) and np.all(got[4][:t0.size] == 1)
        for g, x in zip(got, want):
            np.testing.assert_array_equal(g.view(np.uint32), x.view(np.uint32))


def same_learner(x, y, P):
    for l in range(P):
        x.select(l)
        y.select(l)
        for net in range(4):
            for k in range(3):
                for u, v in zip(x.get_layer(net, k), y.get_layer(net, k)):
                    np.testing.assert_array_equal(u.view(np.uint32), v.view(np.uint32))
        for net in (0, 1):
            for k in range(3):
                for u, v in zip(x.get_grad(net, k), y.get_grad(net, k)):
                    np.testing.assert_array_equal(u.view(np.uint32), v.view(np.uint32))
        assert x.losses() == y.losses()


REGIMES = {   # name: (batch, tensor cores, fused, learners, n, memory capacity)
    "fused120": (120, 0, True, 1, 3, 8192),
    "tiled120": (120, 0, False, 1, 3, 8192),
    "tf32_512": (512, 1, False, 1, 8, 8192),
    "chain8192": (8192, 1, False, 1, 16, 16384),
    "population4": (120, 0, False, 4, 5, 4096),
}


@pytest.mark.parametrize("regime", sorted(REGIMES))
def test_update_equals_materialised_twin(sb, train_series, regime):
    B, tc, fused, P, n, cap = REGIMES[regime]
    kw = dict(batch=B, use_tensor_cores=tc, population=P)
    le, tw = sb.Learner(params=sb.default_ddpg_params(**kw)), sb.Learner(params=sb.default_ddpg_params(**kw))
    assert le.set_fused(fused) == fused and tw.set_fused(fused) == fused
    le.init(7)
    tw.init(7)
    gammas = [0.99, 0.9, 0.95, 0.8][:P]
    mems = [rollout_memory(sb, train_series, cap, 256, 24, 2, 30 + 10 * l) for l in range(P)]
    for l in range(P):
        for x in (le, tw):
            x.select(l).set_hparams(gamma=gammas[l])
            x.set_norm(*mems[l].min_max_buffer(len(mems[l]), rng_mm=1 + l))
    le.select(0)
    tw.select(0)
    seed = 5
    rows = [mems[l].sample_nstep(B, seed=seed + l, n=n, gamma=gammas[l]) for l in range(P)]
    ks = torch.cat([r[5] for r in rows]).cpu().numpy()
    assert ks.max() == n and ks.min() < n, "rows walk whole chains and stop at episode ends"
    twins = []
    for s, a, r, s2, d, _ in rows:
        t = sb.Replay(B)
        t.push(s, a, r, s2, d)
        twins.append(t)
    le.set_nstep(n)
    assert le.get_nstep() == n
    ident = np.tile(np.arange(B, dtype=np.int32), (P, 1, 1))
    if P == 1:
        le.replay(mems[0], rng_rpl=seed)
        tw.replay(twins[0], idx=ident[0])
    else:
        le.replay(mems, rng_rpl=seed)
        tw.replay(twins, idx=ident)
    same_learner(le, tw, P)


def test_prioritized_nstep_equals_twin(sb, train_series):
    B, n, seed, beta = 120, 3, 9, 0.4
    mem = rollout_memory(sb, train_series, 8192, 256, 24, 2, 50)
    mem.enable_priorities()
    le, tw = sb.Learner(), sb.Learner()
    le.init(3)
    tw.init(3)
    for x in (le, tw):
        x.set_norm(*mem.min_max_buffer(len(mem), rng_mm=1))
        x.set_prioritized(0.6, beta, 1e-3)
    le.set_nstep(n)
    idx, _ = mem.sample_prioritized(B, seed=seed, beta=beta)
    idx = idx.cpu().numpy()
    s, a, r, s2, d, k = mem.sample_nstep(B, idx=idx, n=n, gamma=0.99)
    assert k.max().item() == n
    twin = sb.Replay(B)
    twin.push(s, a, r, s2, d)
    twin.enable_priorities()
    le.replay(mem, rng_rpl=seed)
    tw.replay(twin, idx=np.arange(B, dtype=np.int32))
    same_learner(le, tw, 1)
    # the write-back lands on the rows' first records (a record drawn twice keeps the larger priority), nowhere else
    got, pm = mem.priorities()
    tp, tpm = twin.priorities()
    drawn = {}
    for j, i in enumerate(idx):
        drawn[int(i)] = max(drawn.get(int(i), -np.inf), tp[j])
    want = np.ones(len(mem), np.float32)
    want[list(drawn)] = list(drawn.values())
    np.testing.assert_array_equal(got, want)
    assert pm == tpm


def test_n1_ignores_links(sb, train_series):
    rng = np.random.default_rng(6)
    a, b = sb.Replay(3000), sb.Replay(3000).enable_successors()
    w = Walker(rng, 100)
    for _ in range(25):
        x = [dev(v) for v in w.step()]
        a.push(*x)
        b.push(*x)
    la, lb = sb.Learner(), sb.Learner()
    la.init(4)
    lb.init(4)
    for le, m in ((la, a), (lb, b)):
        le.set_norm(*m.min_max_buffer(len(m), rng_mm=2))
        le.set_nstep(1)
        le.replay(m, rng_rpl=8, n_updates=3)
    same_learner(la, lb, 1)


def test_driver_resume_is_bit_identical(sb, train_series, tmp_path):
    n, T = 64, 24

    def make():
        env = sb.Shems(T, train_series, n_envs=n)
        return sb.ddpg.Driver(env, mem_size=3000, ep_length=T, nstep=3), env

    def run(drv, env, episodes):
        for e in episodes:
            drv.episode(env, train=True, rng_ep=e)

    d1, e1 = make()
    assert d1.learner.get_nstep() == 3 and d1.memory.has_successors
    d1.learner.init(3)
    d1.populate_memory()
    d1.min_max_buffer()
    run(d1, e1, [1, 2])
    path = str(tmp_path / "ck.npz")
    sb.tracker.save_checkpoint(path, d1.learner, memories=d1.memory)
    assert len(d1.memory) == d1.memory.capacity
    run(d1, e1, [3, 4])
    d2, e2 = make()
    d2.learner.init(3)
    sb.tracker.load_checkpoint(path, d2.learner, memories=d2.memory)
    run(d2, e2, [3, 4])
    same_learner(d1.learner, d2.learner, 1)
    np.testing.assert_array_equal(d1.memory.successors(), d2.memory.successors())


def test_rejections(sb, train_series):
    rng = np.random.default_rng(2)
    le = sb.Learner()
    le.init(4)
    plain, mem = sb.Replay(500), sb.Replay(500).enable_successors()
    for m in (plain, mem):
        m.push(*[dev(v) for v in Walker(rng, 300).step()])
    for bad in (0, 17, -1):
        with pytest.raises(sb.ShemsError):
            le.set_nstep(bad)
    assert le.get_nstep() == 1
    with pytest.raises(sb.ShemsError):
        plain.successors()
    with pytest.raises(sb.ShemsError):
        plain.set_successors(np.full(300, -1, np.int32))
    with pytest.raises(sb.ShemsError):
        plain.sample_nstep(8, n=2)
    for bad_n in (0, 17):
        with pytest.raises(sb.ShemsError):
            mem.sample_nstep(8, n=bad_n)
    nx = mem.successors()
    for i, v in ((5, 5), (5, 3), (7, 300), (9, -2)):   # itself, an older record, past the end, below -1
        bad = nx.copy()
        bad[i] = v
        with pytest.raises(sb.ShemsError):
            mem.set_successors(bad)
        np.testing.assert_array_equal(mem.successors(), nx)
    le.set_nstep(4)
    before = [le.get_layer(n, k)[0].copy() for n in range(4) for k in range(3)]
    with pytest.raises(sb.ShemsError):
        le.replay(plain, rng_rpl=1)                 # memory without links
    with pytest.raises(sb.ShemsError):
        le.replay_dp(mem)                           # ddpg_update_phase
    with pytest.raises(sb.ShemsError):
        le.replay_fused_dp(mem)                     # ddpg_update_dp
    with pytest.raises(sb.ShemsError):
        le.dp_connect(0, 1, [le.dp_export()])
    env = sb.Shems(8, train_series, n_envs=32)
    env.reset(rng=1)
    with pytest.raises(sb.ShemsError):
        le.episode(env, plain, 4, train=True)
    after = [le.get_layer(n, k)[0] for n in range(4) for k in range(3)]
    for x, y in zip(before, after):
        np.testing.assert_array_equal(x, y)
    pop = sb.Learner(params=sb.default_ddpg_params(population=2))
    pop.set_nstep(2)
    with pytest.raises(sb.ShemsError):
        pop.replay([mem, plain], rng_rpl=1)         # every learner needs links
