"""The lock-step loop of the trimmed rollout kernel against its two-step loop and against the general kernel, bit for bit.

A warp of shems_rollout_lean_kernel whose instances all start on one row runs a loop that dispatches each step to a body compiled
for the row's class (PV covers the demand or not, EV absent or connected); SHEMS_ROLLOUT_LOCKSTEP=0 keeps every warp on the two-step
loop and SHEMS_ROLLOUT_LEAN=0 runs the general kernel.  Each case runs the same seeded sequence all three ways and requires byte-equal
obs, idx, ep_return, reward trajectories and ring contents.  The cases cover the three policies, launches where every warp is in lock
step and where only some are, a partial last warp without a ring, odd step0 and odd T, multi-group envs and a series that holds every
row class and the rows that stay general (departure hour, c_ev = -0.0 and in (-1, 0)) next to rows with PV equal to the demand.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

SWITCHES = [("SHEMS_ROLLOUT_LOCKSTEP", "0"), ("SHEMS_ROLLOUT_LEAN", "0")]


def bits(x):
    x = np.ascontiguousarray(x.cpu().numpy() if torch.is_tensor(x) else np.asarray(x))
    return x.view({4: np.uint32, 8: np.uint64}[x.dtype.itemsize])


def all_ways(monkeypatch, run):
    new = run()
    for var, val in SWITCHES:
        monkeypatch.setenv(var, val)
        ref = run()
        monkeypatch.delenv(var)
        torch.cuda.synchronize()
        assert ref.keys() == new.keys()
        for k in ref:
            assert ref[k].shape == new[k].shape, (var, k)
            bx, by = bits(ref[k]), bits(new[k])
            assert np.array_equal(bx, by), (var, k, int(np.count_nonzero(bx != by)))


def snapshot(out, env, mem, tag=""):
    out[tag + "obs"], out[tag + "idx"] = env.state, env.idx
    if mem is not None and len(mem):
        for name, x in zip(("s", "a", "r", "s2", "done"), mem.get()):
            out[tag + "ring_" + name] = x


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


def every_class_series(sb, nrows=600):
    """a synthetic year slice whose h_countdown cycles through absent, connected, departure, -0.0 and (-1, 0) rows and whose PV
    equals the demand on every fifth row"""
    ser = sb.series.synth_charger98(nrows, seed=5).copy()
    cd = np.array([-1.0, -1.0, 3.0, 2.0, 1.0, 0.0, -1.0, -0.0, 4.0, -0.5, -1.0, 7.0, -1.0], np.float32)
    ser[1] = np.resize(cd, nrows)
    ser[3, ::5] = ser[2, ::5]
    ser[3, 1::3] += 2.5   # more rows where PV covers the demand
    return ser


@pytest.mark.parametrize("policy", ["RANDOM", "RULE", "TAPE"])
@pytest.mark.parametrize("series", ["synth", "every_class"])
def test_lock_step(sb, train_series, monkeypatch, policy, series):
    """every instance starts at row 1 (rng = -1), so every warp is in lock step"""
    pol = getattr(sb, "POLICY_" + policy)
    ser = train_series if series == "synth" else every_class_series(sb)

    def run():
        env = sb.Shems(80, ser, n_envs=256)
        mem = sb.Replay(256 * 64)
        env.reset(rng=-1)
        return rollouts(sb, env, mem, [(pol, 31), (pol, 17), (pol, 24)])   # step0 = 0, 31 (odd), 48; T odd and even

    all_ways(monkeypatch, run)


@pytest.mark.parametrize("policy", ["RANDOM", "RULE"])
def test_some_warps_uniform(sb, monkeypatch, policy):
    """one instance of the second warp starts on another row: that warp runs the two-step loop, the others the lock-step loop"""
    pol = getattr(sb, "POLICY_" + policy)
    ser = every_class_series(sb)
    n = 128
    idx0 = np.ones(n, np.int32)
    idx0[45] = 4
    socb0 = np.linspace(0.0, 6.0, n).astype(np.float32)

    def run():
        env = sb.Shems(60, ser, n_envs=n)
        mem = sb.Replay(n * 64)
        env.reset(idx0=idx0, socb0=socb0)
        idx = env.idx
        assert idx[44] != idx[45] and len(set(idx[:32])) == 1
        return rollouts(sb, env, mem, [(pol, 25), (pol, 30)])

    all_ways(monkeypatch, run)


@pytest.mark.parametrize("policy", ["RANDOM", "RULE", "TAPE"])
def test_partial_last_warp(sb, monkeypatch, policy):
    """N = 1000 without a ring: the last warp has 8 lanes"""
    pol = getattr(sb, "POLICY_" + policy)
    ser = every_class_series(sb)

    def run():
        env = sb.Shems(70, ser, n_envs=1000)
        env.reset(rng=-1)
        return rollouts(sb, env, None, [(pol, 1), (pol, 29), (pol, 30)])

    all_ways(monkeypatch, run)


def test_groups(sb, monkeypatch):
    T = 25
    groups = [(98, 64), (4, 96), (7, 32)]
    ser = np.stack([every_class_series(sb, 300), sb.series.synth_charger98(300, seed=4), sb.series.synth_charger98(300, seed=7)])

    def run():
        env = sb.Shems(3 * T, ser, groups=groups)
        mem = sb.Replay(env.n_envs * 8)
        env.reset(rng=-1)
        return rollouts(sb, env, mem, [(sb.POLICY_RANDOM, T), (sb.POLICY_RULE, T), (sb.POLICY_RANDOM, T)])

    all_ways(monkeypatch, run)
