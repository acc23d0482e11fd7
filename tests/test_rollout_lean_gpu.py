"""The trimmed rollout kernel (shems_rollout_lean_kernel) against the general one, bit for bit.

A rollout from a consistent env with FAST constants, no trace and no obs trajectory takes the trimmed kernel when its ring sink
(if any) stores compact records and N and the ring capacity are multiples of 32; SHEMS_ROLLOUT_LEAN=0 forces the general kernel.
Each case runs the same seeded sequence both ways and requires byte-equal obs, idx, ep_return, reward trajectories and ring
contents (get over all slots and min_max_buffer).  The cases cover the three policies, compact and forced-full records, N a
multiple of 32 and not, a capacity that is not, an unaligned ring head, a ring wrap inside one launch, odd step0 and odd T (the
kernel draws one Philox block per step pair), multi-group envs, training-shaped windows and the set_state fallback.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def bits(x):
    x = np.ascontiguousarray(x.cpu().numpy() if torch.is_tensor(x) else np.asarray(x))
    return x.view({4: np.uint32, 8: np.uint64}[x.dtype.itemsize])


def both(monkeypatch, run):
    monkeypatch.setenv("SHEMS_ROLLOUT_LEAN", "0")
    ref = run()
    monkeypatch.delenv("SHEMS_ROLLOUT_LEAN")
    new = run()
    torch.cuda.synchronize()
    assert ref.keys() == new.keys()
    for k in ref:
        assert ref[k].shape == new[k].shape, k
        bx, by = bits(ref[k]), bits(new[k])
        assert np.array_equal(bx, by), (k, int(np.count_nonzero(bx != by)))


def snapshot(out, env, mem, tag=""):
    out[tag + "obs"], out[tag + "idx"] = env.state, env.idx
    if mem is not None and len(mem):
        for name, x in zip(("s", "a", "r", "s2", "done"), mem.get()):
            out[tag + "ring_" + name] = x
        for i, x in enumerate(mem.min_max_buffer(len(mem), rng_mm=2)):
            out[tag + "minmax%d" % i] = x


def rollouts(sb, env, mem, plan, seed=11):
    """plan: [(policy, T)]; returns every output of every rollout and the final state"""
    out = {}
    for j, (pol, T) in enumerate(plan):
        tape = None
        if pol == sb.POLICY_TAPE:
            g = torch.Generator(device="cuda").manual_seed(seed + j)
            tape = torch.rand((T, 2, env.n_envs), generator=g, device="cuda") * 2 - 1
        res = env.rollout(pol, T, seed=seed + j, tape=tape, tape_unscaled=tape is not None, replay=mem, want_reward=True)
        for k, v in res.items():
            out["%d_%s" % (j, k)] = v.clone()
        snapshot(out, env, None, "%d_" % j)
    snapshot(out, env, mem)
    return out


@pytest.mark.parametrize("compact", [True, False])
@pytest.mark.parametrize("policy", ["RANDOM", "RULE", "TAPE"])
@pytest.mark.parametrize("n", [256, 1000])
def test_policies(sb, train_series, monkeypatch, policy, compact, n):
    if not compact:
        monkeypatch.setenv("SHEMS_RING_COMPACT", "0")
    pol = getattr(sb, "POLICY_" + policy)

    def run():
        env = sb.Shems(80, train_series, n_envs=n)
        mem = sb.Replay(n * 64)
        env.reset(rng=3)
        return rollouts(sb, env, mem, [(pol, 31), (pol, 17), (pol, 24)])   # step0 = 0, 31 (odd), 48; T odd and even

    both(monkeypatch, run)


@pytest.mark.parametrize("policy", ["RANDOM", "RULE"])
def test_returns_only(sb, train_series, monkeypatch, policy):
    pol = getattr(sb, "POLICY_" + policy)

    def run():
        env = sb.Shems(60, train_series, n_envs=320)
        env.reset(rng=2)
        return rollouts(sb, env, None, [(pol, 1), (pol, 29), (pol, 30)])

    both(monkeypatch, run)


def push_random(mem, n, seed):
    rng = np.random.default_rng(seed)
    t = [torch.as_tensor(rng.normal(size=sh).astype(np.float32), device="cuda") for sh in ((9, n), (2, n), (n,), (9, n))]
    mem.push(*t)


@pytest.mark.parametrize("cap_extra", [0, 7])
def test_unaligned_head(sb, train_series, monkeypatch, cap_extra):
    """an odd push leaves the head off a 32-slot tile; cap_extra = 7 makes the capacity not a multiple of 32"""
    n, T = 128, 21

    def run():
        env = sb.Shems(T, train_series, n_envs=n)
        mem = sb.Replay(n * T + 64 + cap_extra)
        push_random(mem, 37, 1)
        env.reset(rng=4)
        return rollouts(sb, env, mem, [(sb.POLICY_RANDOM, T)])

    both(monkeypatch, run)


@pytest.mark.parametrize("head", [0, 45])
def test_wrap_inside_one_launch(sb, train_series, monkeypatch, head):
    n, T = 160, 71   # 11360 transitions through 16 x 160 slots

    def run():
        env = sb.Shems(T + 2, train_series, n_envs=n)
        mem = sb.Replay(16 * n)
        if head:
            push_random(mem, head, 5)
        env.reset(rng=5)
        return rollouts(sb, env, mem, [(sb.POLICY_RANDOM, 1), (sb.POLICY_RANDOM, T)])

    both(monkeypatch, run)


def test_groups(sb, monkeypatch):
    T = 25
    groups = [(98, 64), (4, 96), (7, 32)]
    ser = np.stack([sb.series.synth_charger98(4320, seed=s) for s in (98, 4, 7)])

    def run():
        env = sb.Shems(3 * T, ser, groups=groups)
        mem = sb.Replay(env.n_envs * 8)
        env.reset(rng=8)
        return rollouts(sb, env, mem, [(sb.POLICY_RANDOM, T), (sb.POLICY_RULE, T), (sb.POLICY_RANDOM, T)])

    both(monkeypatch, run)


def test_training_windows(sb, monkeypatch):
    """72-step rollouts from random windows of a 4320-row series, as training fills its memory"""
    ser = sb.series.synth_charger98(4320, seed=98)

    def run():
        env = sb.Shems(72, ser, n_envs=2048)
        mem = sb.Replay(2048 * 72 * 2)
        out = {}
        for ep in range(3):
            env.reset(rng=ep + 1)
            for k, v in rollouts(sb, env, mem, [(sb.POLICY_RANDOM, 72)], seed=ep).items():
                out["%d_%s" % (ep, k)] = v
        return out

    both(monkeypatch, run)


def test_set_state_then_consistent(sb, train_series, monkeypatch):
    """after set_state the general kernel runs (s[2..8] need not be series rows); the rollout after it is consistent again"""
    n = 96
    rng = np.random.default_rng(0)
    idx = rng.integers(1, 4000, n).astype(np.int32)
    obs = rng.uniform(0, 1, (9, n)).astype(np.float32)

    def run():
        env = sb.Shems(40, train_series, n_envs=n)
        mem = sb.Replay(n * 64)
        env.set_state(obs, idx)
        return rollouts(sb, env, mem, [(sb.POLICY_RANDOM, 9), (sb.POLICY_RANDOM, 13)])

    both(monkeypatch, run)
