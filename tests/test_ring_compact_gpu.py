"""Compact replay records (csrc/ring.cuh): a rollout from a series-consistent env stores 8 words per transition and names the
series rows that hold the other 14 fields.  Every reader must hand back exactly the bits a full 22-field record gives.

Each case fills two rings the same way, one with SHEMS_RING_COMPACT=0 (full records only) and one with compact records allowed,
and requires byte-equal results from replay_get, sample (caller indices and Philox), min_max_buffer and the learner parameters
after a few updates on the cluster-fused path, the tiled path and a small population.
"""
import gc

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

N_UPDATES = 3


def bits(x):
    x = np.ascontiguousarray(x.cpu().numpy() if torch.is_tensor(x) else x)
    return x.view(np.uint32 if x.dtype == np.float32 else np.uint64)


def assert_same(x, y, what):
    assert x.shape == y.shape, what
    bx, by = bits(x), bits(y)
    assert np.array_equal(bx, by), (what, int(np.count_nonzero(bx != by)))


def learned(sb, mems, fused=None, population=0):
    """layers of all four nets after N_UPDATES replay() calls from `mems` (normalised by the ring's own min/max)"""
    mn, mx = mems[0].min_max_buffer(len(mems[0]), rng_mm=1)
    if population:
        le = sb.Learner(params=sb.default_ddpg_params(population=population))
    else:
        le = sb.Learner()
        le.set_fused(fused)
    le.init(11)
    for l in range(max(population, 1)):
        le.select(l).set_norm(mn, mx)
    le.replay(list(mems) if population else mems[0], rng_rpl=5, n_updates=N_UPDATES)
    out = []
    for l in range(max(population, 1)):
        le.select(l)
        for net in range(4):
            for k in range(3):
                w, b = le.get_layer(net, k)
                out += [w, b]
    le.close()
    return out


def compare(sb, full, compact, learn=True):
    for name, x, y in zip(("s", "a", "r", "s2", "done"), full.get(), compact.get()):
        assert_same(x, y, "get " + name)
    n = len(full)
    assert len(compact) == n
    idx = np.random.default_rng(3).integers(0, n, 257).astype(np.int32)
    for name, x, y in zip(("s", "a", "r", "s2", "done"), full.sample(257, idx=idx), compact.sample(257, idx=idx)):
        assert_same(x, y, "sample(idx) " + name)
    for name, x, y in zip(("s", "a", "r", "s2", "done"), full.sample(300, rng_dt=9), compact.sample(300, rng_dt=9)):
        assert_same(x, y, "sample(philox) " + name)
    for x, y in zip(full.min_max_buffer(n, rng_mm=2), compact.min_max_buffer(n, rng_mm=2)):
        assert_same(x, y, "min_max_buffer")
    for x, y in zip(full.min_max_buffer(len(idx), idx=idx), compact.min_max_buffer(len(idx), idx=idx)):
        assert_same(x, y, "min_max_buffer(idx)")
    if learn:
        for kw in (dict(fused=True), dict(fused=False), dict(population=2)):
            for i, (x, y) in enumerate(zip(learned(sb, [full] * max(kw.get("population", 1), 1), **kw),
                                           learned(sb, [compact] * max(kw.get("population", 1), 1), **kw))):
                assert_same(x, y, "parameters %s #%d" % (kw, i))


def both(monkeypatch, fill):
    """(ring filled with full records only, ring filled with compact records allowed)"""
    monkeypatch.setenv("SHEMS_RING_COMPACT", "0")
    full = fill()
    monkeypatch.delenv("SHEMS_RING_COMPACT")
    compact = fill()
    torch.cuda.synchronize()
    assert full.series_copies == 0
    return full, compact


def push_random(mem, n, seed):
    rng = np.random.default_rng(seed)
    t = [torch.as_tensor(rng.normal(size=sh).astype(np.float32), device="cuda") for sh in ((9, n), (2, n), (n,), (9, n))]
    mem.push(*t)


@pytest.mark.parametrize("policy", ["RANDOM", "RULE", "TAPE"])
def test_policies(sb, train_series, monkeypatch, policy):
    n, T = 200, 30
    pol = getattr(sb, "POLICY_" + policy)
    tape = None
    if policy == "TAPE":
        g = torch.Generator(device="cuda").manual_seed(4)
        tape = torch.rand((T, 2, n), generator=g, device="cuda") * 2 - 1

    def fill():
        env = sb.Shems(T, train_series, n_envs=n)
        mem = sb.Replay(n * T)
        env.reset(rng=3)
        env.rollout(pol, T, seed=5, tape=tape, tape_unscaled=tape is not None, replay=mem)
        return mem

    full, compact = both(monkeypatch, fill)
    assert compact.series_copies == 1
    compare(sb, full, compact)


@pytest.mark.parametrize("per_group", [True, False])
def test_groups(sb, train_series, monkeypatch, per_group):
    T = 24
    groups = [(98, 70), (4, 90), (7, 33)]
    ser = np.stack([sb.series.synth_charger98(4320, seed=s) for s in (98, 4, 7)]) if per_group else train_series

    def fill():
        env = sb.Shems(2 * T, ser, groups=groups)
        mem = sb.Replay(env.n_envs * T * 2)
        env.reset(rng=8)
        env.rollout(sb.POLICY_RANDOM, T, seed=2, replay=mem)
        env.rollout(sb.POLICY_RULE, T, replay=mem)
        return mem

    full, compact = both(monkeypatch, fill)
    assert compact.series_copies == (3 if per_group else 1)
    compare(sb, full, compact)


def test_unaligned_head_after_pushes(sb, train_series, monkeypatch):
    n, T = 96, 20

    def fill():
        env = sb.Shems(T, train_series, n_envs=n)
        mem = sb.Replay(n * T + 100)
        push_random(mem, 37, 1)
        push_random(mem, 12, 2)
        env.reset(rng=4)
        env.rollout(sb.POLICY_RANDOM, T, seed=6, replay=mem)
        return mem

    full, compact = both(monkeypatch, fill)
    assert compact.series_copies == 1
    compare(sb, full, compact)


def test_wrap_with_capacity_multiple_of_envs(sb, train_series, monkeypatch):
    n, T = 160, 70   # 11200 transitions through 16 x 160 slots, as the benchmark wraps its ring

    def fill():
        env = sb.Shems(T, train_series, n_envs=n)
        mem = sb.Replay(16 * n)
        env.reset(rng=5)
        env.rollout(sb.POLICY_RANDOM, T, seed=7, replay=mem)
        return mem

    full, compact = both(monkeypatch, fill)
    assert compact.series_copies == 1 and len(compact) == 16 * n
    compare(sb, full, compact)


def test_set_state_falls_back_to_full_records(sb, train_series, monkeypatch):
    n, T = 64, 12
    rng = np.random.default_rng(0)
    idx = rng.integers(1, 4000, n).astype(np.int32)
    obs = rng.uniform(0, 1, (9, n)).astype(np.float32)   # state fields 2..8 unrelated to the series rows

    def fill():
        env = sb.Shems(T, train_series, n_envs=n)
        mem = sb.Replay(n * T * 2)
        env.set_state(obs, idx)
        env.rollout(sb.POLICY_RANDOM, T, seed=1, replay=mem)
        return mem

    full, compact = both(monkeypatch, fill)
    assert compact.series_copies == 0
    compare(sb, full, compact, learn=False)
    s, _, _, _, _ = compact.get()
    assert_same(s[:, :n], obs, "the injected state is what the first records hold")


def test_pushes_overwrite_compact_slots(sb, train_series, monkeypatch):
    n, T = 128, 8

    def fill():
        env = sb.Shems(64, train_series, n_envs=n)
        mem = sb.Replay(n * 4)
        env.reset(rng=6)
        env.rollout(sb.POLICY_RANDOM, T, seed=3, replay=mem)    # every slot compact (the ring wraps twice)
        push_random(mem, 50, 3)                                  # full records over the oldest compact slots
        env.rollout(sb.POLICY_RULE, 2, replay=mem)
        push_random(mem, 31, 4)
        return mem

    full, compact = both(monkeypatch, fill)
    assert compact.series_copies == 1
    compare(sb, full, compact)


def test_readable_after_env_is_destroyed(sb, monkeypatch):
    n, T = 256, 24

    def fill():
        ser = sb.series.synth_charger98(2000, seed=21)
        env = sb.Shems(T, ser, n_envs=n)
        mem = sb.Replay(n * T)
        env.reset(rng=9)
        env.rollout(sb.POLICY_RANDOM, T, seed=9, replay=mem)
        env.close()
        del env, ser
        gc.collect()
        # a new env may get the freed series' address: its records must not be mistaken for the old env's
        other = sb.Shems(T, sb.series.synth_charger98(2000, seed=22), n_envs=n)
        other.reset(rng=1)
        other.rollout(sb.POLICY_RANDOM, 2, seed=1, replay=mem)
        other.close()
        return mem

    full, compact = both(monkeypatch, fill)
    assert compact.series_copies == 2
    compare(sb, full, compact)
