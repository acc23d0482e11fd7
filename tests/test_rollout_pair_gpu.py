"""The pair kernel of the rollout (two instances per thread when every instance stands on the same row) against the trimmed kernel
and against the general kernel, bit for bit.

SHEMS_ROLLOUT_PAIR=2 takes the pair kernel wherever it applies, whatever the grid size; SHEMS_ROLLOUT_PAIR=0 runs the trimmed
kernel's lock-step loop and SHEMS_ROLLOUT_LEAN=0 the general kernel.  Each case runs the same seeded sequence all three ways, requires
byte-equal obs, idx, ep_return, reward trajectories and ring contents, and checks through the library's launch counter how many
launches took the pair kernel, so that a case cannot pass by never pairing (or by pairing where it must not).
"""
import numpy as np
import pytest

from test_rollout_lockstep_gpu import bits, every_class_series, rollouts

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

REFS = [("SHEMS_ROLLOUT_PAIR", "0"), ("SHEMS_ROLLOUT_LEAN", "0")]


def pair_launches(sb):
    return int(sb._lib.lib().shems_rollout_pair_launches())


def all_ways(sb, monkeypatch, run, paired):
    """run() with the pair kernel forced on wherever it applies, then with each reference; `paired` launches must take it"""
    monkeypatch.setenv("SHEMS_ROLLOUT_PAIR", "2")
    c0 = pair_launches(sb)
    new = run()
    assert pair_launches(sb) - c0 == paired
    monkeypatch.delenv("SHEMS_ROLLOUT_PAIR")
    for var, val in REFS:
        monkeypatch.setenv(var, val)
        c0 = pair_launches(sb)
        ref = run()
        assert pair_launches(sb) == c0
        monkeypatch.delenv(var)
        torch.cuda.synchronize()
        assert ref.keys() == new.keys()
        for k in ref:
            assert ref[k].shape == new[k].shape, (var, k)
            bx, by = bits(ref[k]), bits(new[k])
            assert np.array_equal(bx, by), (var, k, int(np.count_nonzero(bx != by)))


@pytest.mark.parametrize("policy", ["RANDOM", "RULE", "TAPE"])
@pytest.mark.parametrize("series", ["synth", "every_class"])
def test_pair(sb, train_series, monkeypatch, policy, series):
    """rng = -1: every instance on row 1; step0 = 0, 31 (odd), 48 with odd and even T"""
    pol = getattr(sb, "POLICY_" + policy)
    ser = train_series if series == "synth" else every_class_series(sb)

    def run():
        env = sb.Shems(80, ser, n_envs=256)
        mem = sb.Replay(256 * 64)
        env.reset(rng=-1)
        return rollouts(sb, env, mem, [(pol, 31), (pol, 17), (pol, 24)])

    all_ways(sb, monkeypatch, run, paired=3)


@pytest.mark.parametrize("ring", [True, False])
def test_groups(sb, monkeypatch, ring):
    """groups of 33, 64 and 31 instances: only the middle one has an even count, and it starts at instance 33 — paired without a
    ring, not with one (its first slot is odd)"""
    T = 25
    groups = [(98, 33), (4, 64), (7, 31)]
    ser = np.stack([every_class_series(sb, 300), sb.series.synth_charger98(300, seed=4), sb.series.synth_charger98(300, seed=7)])

    def run():
        env = sb.Shems(3 * T, ser, groups=groups)
        mem = sb.Replay(env.n_envs * 8) if ring else None
        env.reset(rng=-1)
        return rollouts(sb, env, mem, [(sb.POLICY_RANDOM, T), (sb.POLICY_RULE, T), (sb.POLICY_RANDOM, T)])

    all_ways(sb, monkeypatch, run, paired=0 if ring else 3)


def test_even_groups(sb, monkeypatch):
    T = 24
    groups = [(98, 64), (4, 96), (7, 32)]
    ser = np.stack([every_class_series(sb, 300), sb.series.synth_charger98(300, seed=4), sb.series.synth_charger98(300, seed=7)])

    def run():
        env = sb.Shems(3 * T, ser, groups=groups)
        mem = sb.Replay(env.n_envs * 8)
        env.reset(rng=-1)
        return rollouts(sb, env, mem, [(sb.POLICY_RANDOM, T), (sb.POLICY_TAPE, T + 1), (sb.POLICY_RANDOM, T - 1)])

    all_ways(sb, monkeypatch, run, paired=9)


@pytest.mark.parametrize("pushed,paired", [(1, 0), (2, 3)])
def test_ring_head(sb, monkeypatch, pushed, paired):
    """`pushed` transitions go into the ring first: an odd head takes the trimmed kernel, an even one pairs; the ring of 8 N slots
    wraps inside the second and third launches"""
    n = 128
    ser = every_class_series(sb)

    def run():
        env = sb.Shems(90, ser, n_envs=n)
        mem = sb.Replay(n * 8)
        g = torch.Generator(device="cuda").manual_seed(3)
        s, s2 = torch.rand((9, pushed), generator=g, device="cuda"), torch.rand((9, pushed), generator=g, device="cuda")
        mem.push(s, torch.rand((2, pushed), generator=g, device="cuda"), torch.rand(pushed, generator=g, device="cuda"), s2)
        env.reset(rng=-1)
        return rollouts(sb, env, mem, [(sb.POLICY_RANDOM, 5), (sb.POLICY_RANDOM, 21), (sb.POLICY_RULE, 30)])

    all_ways(sb, monkeypatch, run, paired=paired)


@pytest.mark.parametrize("differ", [False, True])
def test_host_draws(sb, monkeypatch, differ):
    """reset with host draws: every idx0 equal pairs, one differing row does not"""
    n = 128
    ser = every_class_series(sb)
    idx0 = np.full(n, 7, np.int32)
    if differ:
        idx0[77] = 9
    socb0 = np.linspace(0.0, 6.0, n).astype(np.float32)

    def run():
        env = sb.Shems(60, ser, n_envs=n)
        mem = sb.Replay(n * 64)
        env.reset(idx0=idx0, socb0=socb0)
        assert len(set(env.idx)) == (2 if differ else 1)
        return rollouts(sb, env, mem, [(sb.POLICY_RANDOM, 25), (sb.POLICY_RULE, 30)])

    all_ways(sb, monkeypatch, run, paired=0 if differ else 2)


def test_device_draws(sb, monkeypatch):
    """a Philox reset with more than one admissible start row does not pair"""
    ser = every_class_series(sb)

    def run():
        env = sb.Shems(60, ser, n_envs=128)
        env.reset(rng=5)
        return rollouts(sb, env, None, [(sb.POLICY_RANDOM, 25)])

    all_ways(sb, monkeypatch, run, paired=0)


@pytest.mark.parametrize("differ", [False, True])
def test_set_state(sb, monkeypatch, differ):
    """set_state leaves the env inconsistent, so its first rollout runs the general kernel; the second pairs when every row is equal"""
    n = 64
    ser = every_class_series(sb)
    rng = np.random.default_rng(4)
    idx = np.full(n, 11, np.int32)
    if differ:
        idx[5] = 12
    obs = rng.uniform(0.0, 1.0, (9, n)).astype(np.float32)

    def run():
        env = sb.Shems(60, ser, n_envs=n)
        mem = sb.Replay(n * 64)
        env.reset(rng=-1)
        env.set_state(obs, idx)
        return rollouts(sb, env, mem, [(sb.POLICY_RANDOM, 9), (sb.POLICY_RANDOM, 14)])

    all_ways(sb, monkeypatch, run, paired=0 if differ else 1)


@pytest.mark.parametrize("n,paired", [(1001, 0), (1000, 3)])
def test_no_ring(sb, monkeypatch, n, paired):
    """without a ring: an odd count does not pair; 1000 instances pair into 500 threads (a partial last warp)"""
    ser = every_class_series(sb)

    def run():
        env = sb.Shems(70, ser, n_envs=n)
        env.reset(rng=-1)
        return rollouts(sb, env, None, [(sb.POLICY_RANDOM, 1), (sb.POLICY_TAPE, 29), (sb.POLICY_RULE, 30)])

    all_ways(sb, monkeypatch, run, paired=paired)
