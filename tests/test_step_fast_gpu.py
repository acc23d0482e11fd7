"""The FAST instantiations of the step and rollout kernels against the generic ones, bit for bit.

A launch without a trace takes the FAST instantiation when the constants allow it; asking for a trace takes the generic one.  FAST
takes the Float32 decisions against Float64 constants (the battery rate R, 0.95 smax) in FP32 against thresholds the host rounded,
decodes random actions without Float64 and divides the Float32 quotients by eta and span through Float64 without a guard, where the
generic path uses the guarded Float32 sequence.  The states are injected with set_state and include the boundaries of those rewrites:
Soc_b - smin at 0, subnormal and around 2^-60, the charge request and pv at RD32(R), RU32(R) and one ulp either side, B at
+-0.01f +- 1 ulp, Soc_b at 1e-3f +- 1 ulp, and the seeded cases of tests/lu1_cases.py that reach every flow leaf.
"""
import numpy as np
import pytest

import lu1_cases as Cs

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

F32 = np.float32
T = 72


def ulps(x):
    x = F32(x)
    return [np.nextafter(x, F32(-np.inf)), x, np.nextafter(x, F32(np.inf))]


def rd_ru(c):
    f = F32(c)
    lo = f if float(f) <= c else np.nextafter(f, F32(-np.inf))
    hi = f if float(f) >= c else np.nextafter(f, F32(np.inf))
    return lo, hi


def soc_for(target, base):
    """Float32 Soc_b values s near base - target for which base - s (one Float32 rounding) equals target exactly"""
    out = []
    s0 = F32(base - F32(target))
    for k in range(-8, 9):
        s = F32(s0)
        for _ in range(abs(k)):
            s = np.nextafter(s, F32(np.inf) if k > 0 else F32(-np.inf))
        if F32(base - s) == F32(target) and 0 <= s:
            out.append(s)
    return out


def boundary_states(P, series, idx_max, rng):
    """[9][n] states and [n] actions at the boundaries of the FP32 rewrites"""
    smax, loss, oml = F32(P.b_soc_max), F32(P.b_loss), F32(1) - F32(P.b_loss)
    R = float(P.b_rate_max)
    socs, acts, pvs = [], [], []
    tiny = [F32(0), F32(1e-45), F32(1e-40), F32(2.0 ** -126)] + ulps(2.0 ** -60) + ulps(2.0 ** -59) + ulps(1e-3) + ulps(2.0 ** -100)
    for s in tiny:  # Soc_b - smin at 0, subnormal, around 2^-60 (smin = 0), Soc_b around 1e-3f
        for bt in (F32(0), F32(0.5), F32(1)):
            socs.append(s); acts.append(bt); pvs.append(F32(rng.uniform(-3, 3)))
    for thr in rd_ru(R):
        for t in ulps(thr):
            # charge request h = (Bt*span + smin - Soc_b) + loss at t (Bt = 1): Soc_b = span + loss - t
            for s in soc_for(F32(t) - loss, F32(smax)):
                for pv in list(ulps(thr)) + [F32(t), F32(0.5), F32(-0.5)]:
                    socs.append(s); acts.append(F32(1)); pvs.append(pv)
            # discharge request oml * Soc_b at t
            s = F32(F32(t) / oml)
            for s2 in ulps(s):
                socs.append(s2); acts.append(F32(0)); pvs.append(F32(-1))
            # pv at t against the rate cap with a large charge request
            socs.append(F32(0.25)); acts.append(F32(1)); pvs.append(F32(t))
    for b in ulps(0.01) + ulps(-0.01):  # B = Bc = pv (small positive) or B = Bd = -oml * Soc_b
        if b > 0:
            socs.append(F32(0.5)); acts.append(F32(1)); pvs.append(b)
        else:
            for s in ulps(F32(-b / oml)):
                socs.append(s); acts.append(F32(0)); pvs.append(F32(-1))
    n = len(socs)
    idx = rng.integers(1, idx_max, size=n).astype(np.int32)
    obs = np.zeros((9, n), F32)
    obs[1:] = series[:, idx - 1]
    obs[0] = socs
    obs[1] = 1.0
    obs[2] = -1.0  # no EV connected: EV = 0, so pv = (g_e - d_e) exactly when d_e = 0
    obs[3] = np.where(np.array(pvs) >= 0, 0.0, -np.array(pvs)).astype(F32)
    obs[4] = np.where(np.array(pvs) >= 0, np.array(pvs), 0.0).astype(F32)
    a = np.stack([np.array(acts, F32), np.full(n, 0.5, F32)])
    return obs, idx, a


def all_states(P, series, idx_max, seed):
    rng = np.random.default_rng(seed)
    obs_b, idx_b, a_b = boundary_states(P, series, idx_max, rng)
    cases = Cs.make_cases(series, 20000, seed=seed, charger_id=98)
    keep = cases["track"] >= 0  # the FAST path runs action(env, a); track < 0 steps always carry a trace
    obs_c = cases["state"][keep].T.copy()
    idx_c = np.minimum(cases["idx"][keep], idx_max).astype(np.int32)
    a_c = cases["a"][keep].T.copy()
    return (np.concatenate([obs_b, obs_c], 1), np.concatenate([idx_b, idx_c]), np.concatenate([a_b, a_c], 1))


@pytest.mark.parametrize("charger_id", [98, 4])  # R = 3.3 and R = 4.6 (neither is a Float32 value)
def test_step_fast_equals_generic(sb, O, train_series, charger_id):
    P = O.params_for_charger(charger_id)
    obs, idx, a = all_states(P, train_series, train_series.shape[1] - 1, seed=charger_id)
    n = obs.shape[1]
    out = []
    for track in (0, 1):  # 0: no trace -> FAST; 1: trace -> generic
        env = sb.Shems(T, train_series, n_envs=n, charger_id=charger_id)
        env.set_state(obs, idx)
        r64 = torch.empty(n, dtype=torch.float64, device="cuda")
        res = env.step(torch.as_tensor(a, device="cuda"), track=track, reward64_out=r64)
        out.append((res[0].cpu().numpy().copy(), res[1].cpu().numpy().copy(), r64.cpu().numpy()))
    (r_f, s_f, r64_f), (r_g, s_g, r64_g) = out
    assert s_f.tobytes() == s_g.tobytes()
    assert r_f.tobytes() == r_g.tobytes()
    assert r64_f.tobytes() == r64_g.tobytes()


@pytest.mark.parametrize("charger_id", [98, 4])
@pytest.mark.parametrize("policy", ["rule", "random", "tape"])
def test_rollout_fast_equals_generic(sb, O, train_series, charger_id, policy):
    P = O.params_for_charger(charger_id)
    obs, idx, _ = all_states(P, train_series, train_series.shape[1] - T - 1, seed=7 + charger_id)
    n = obs.shape[1]
    pol = dict(rule=sb.POLICY_RULE, random=sb.POLICY_RANDOM, tape=sb.POLICY_TAPE)[policy]
    raw = np.random.default_rng(5).uniform(-1, 1, (T, 2, n)).astype(F32)
    raw[:, :, ::7] = np.array([-1.0, 1.0], F32)[:, None]
    res = []
    for trace in (False, True):  # FAST vs generic
        env = sb.Shems(T, train_series, n_envs=n, charger_id=charger_id)
        env.set_state(obs, idx)
        mem = sb.Replay(T * n)
        got = env.rollout(pol, T, seed=11, tape=torch.as_tensor(raw, device="cuda") if policy == "tape" else None, replay=mem,
                          want_trace=trace, want_return=True, tape_unscaled=True)
        res.append((env.state, env.idx, got["ep_return"].cpu().numpy(), [x.tobytes() for x in mem.get()]))
    (s_f, i_f, e_f, m_f), (s_g, i_g, e_g, m_g) = res
    assert s_f.tobytes() == s_g.tobytes()
    assert np.array_equal(i_f, i_g)
    assert e_f.tobytes() == e_g.tobytes()
    assert m_f == m_g
