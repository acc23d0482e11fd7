"""Population-based training (ddpg_exploit, Learner.exploit, PopulationDriver.run_episodes(pbt=...)).

The decision (ranks, top and bottom sets, the Philox draw of the source) is restated here in numpy with the oracle's Philox and
compared exactly; the copy is compared bit for bit with ddpg_get_state of the source before the call, and a population trained after
an exploit is compared bit for bit with a twin that received the same states through ddpg_set_state / ddpg_set_hparams."""
import copy
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

STREAM_PBT = 0x5042
NET_ACTOR_BEST = 4
SMALL = dict(l1=48, l2=64)
HP = ("lr_actor", "lr_critic", "gamma", "tau", "noise_scale")


def _memory(sb, series, n=16, T=72, seed=2, capacity=None):
    env = sb.Shems(T, series, n_envs=n)
    mem = sb.Replay(capacity or n * T)
    env.reset(rng=seed)
    env.rollout(sb.POLICY_RANDOM, T, seed=seed, replay=mem, want_return=False)
    return mem


def _population(sb, mems, **kw):
    le = sb.Learner(params=sb.default_ddpg_params(population=len(mems), **kw))
    le.init(21)
    for l, m in enumerate(mems):
        le.select(l).set_norm(*m.min_max_buffer(len(m), rng_mm=l))
    le.select(0)
    return le


def _restate(O, score, sizes, frac, seed, rnd):
    """parent [P] and the second Philox word of every replaced learner, from the rule as the header states it"""
    P = len(score)
    parent, w1 = np.full(P, -1, np.int64), np.zeros(P, np.uint32)
    g0 = 0
    for m in sizes:
        idx = np.arange(g0, g0 + m)
        key = np.where(np.isnan(score[idx]), -np.inf, score[idx])
        order = idx[np.lexsort((idx, -key))]            # descending key, ties to the lower index
        k = int(np.floor(frac * m))
        for d in (order[m - k:] if k > 0 else []):
            w = (C.c_uint32 * 4)()
            O.lib().oracle_philox(seed, int(d), rnd, STREAM_PBT, w)
            parent[d], w1[d] = order[(int(w[0]) * k) >> 32], w[1]
        g0 += m
    return parent, w1


def _perturbed(hp, keys, w1, factors):
    out = dict(hp)
    for j, name in enumerate(HP):
        if name in keys:
            x = np.float32(hp[name]) * np.float32(factors[1] if (int(w1) >> j) & 1 else factors[0])
            out[name] = float(min(x, np.float32(1.0)) if name in ("gamma", "tau") else x)
    return out


def _all(le, mems=None):
    """everything a learner owns that the tests look at, for every learner"""
    P = le.population
    snap = []
    for l in range(P):
        le.select(l)
        st, opt = le.get_state()
        best = [le.get_layer(NET_ACTOR_BEST, k) for k in range(3)]
        snap.append(dict(state=st, opt=opt, hp=le.get_hparams(), best=best, mem=mems[l].get() if mems else None))
    le.select(0)
    return snap, le.best()


def _same(a, b, what):
    np.testing.assert_array_equal(a["state"], b["state"], err_msg=what)
    np.testing.assert_array_equal(a["opt"], b["opt"], err_msg=what)


def _trained(sb, train_series, P, seed=60, **kw):
    """a population whose learners differ in weights, norm, hyper-parameters and best slots, after a few updates"""
    mems = [_memory(sb, train_series, seed=seed + l) for l in range(P)]
    le = _population(sb, mems, **kw)
    rng = np.random.default_rng(seed)
    for l in range(P):
        le.select(l).set_hparams(lr_actor=float(rng.uniform(1e-5, 1e-3)), lr_critic=float(rng.uniform(1e-4, 1e-2)),
                                 gamma=float(rng.uniform(0.9, 0.999)), tau=float(rng.uniform(1e-3, 1e-2)), noise_scale=float(rng.uniform(0.1, 2)))
    le.select(0)
    le.replay(mems, rng_rpl=5, n_updates=3)
    le.keep_best(torch.as_tensor(rng.normal(0, 1, P * 3), device="cuda"), 3, 7)
    le.replay(mems, rng_rpl=6, n_updates=2)
    return le, mems


@pytest.mark.parametrize("sizes", [[5, 1, 2, 4], [4, 2, 6], None])
def test_decision_matches_restatement(sb, O, train_series, sizes):
    """parent equals the restated rank / sets / draw for random scores with ties, NaN and -inf, unequal groups (one of size 1,
    one where k = 0 at frac 0.25), frac 0.5 with even m, several seeds and rounds; groups=None is one group of all P."""
    P = 12
    le = _population(sb, [_memory(sb, train_series, seed=80 + l, n=4) for l in range(P)], batch=32, **SMALL)
    rng = np.random.default_rng(len(sizes or []))
    for trial, (frac, seed, rnd) in enumerate([(0.25, 0, 0), (0.5, 7, 3), (0.34, 2**40 + 3, 2**31 + 5), (0.5, 99, 1), (0.4, 12345, 17)]):
        score = rng.choice([-3.0, -1.5, 0.0, -0.0, 2.0, np.nan, -np.inf], P) if trial % 2 else rng.normal(0, 1, P)
        score[rng.integers(0, P)] = np.nan
        parent = le.exploit(torch.as_tensor(score, device="cuda"), frac, seed=seed, round=rnd, groups=sizes).cpu().numpy()
        want, _ = _restate(O, score, sizes or [P], frac, seed, rnd)
        np.testing.assert_array_equal(parent, want, err_msg=str((trial, frac, seed, rnd)))
        if frac == 0.5 and sizes == [4, 2, 6]:
            assert (parent >= 0).sum() == 2 + 1 + 3
    assert (want >= 0).any()


def test_frac_zero_changes_nothing(sb, train_series):
    P = 4
    le, mems = _trained(sb, train_series, P, batch=32, **SMALL)
    before, best0 = _all(le, mems)
    score = torch.as_tensor(np.arange(P, dtype=np.float64), device="cuda")
    parent = le.exploit(score, 0.0, keys=HP, seed=3, round=1)
    assert (parent.cpu().numpy() == -1).all()
    after, best1 = _all(le, mems)
    for l in range(P):
        _same(before[l], after[l], l)
        assert before[l]["hp"] == after[l]["hp"]
    np.testing.assert_array_equal(best0[0], best1[0])
    np.testing.assert_array_equal(best0[1], best1[1])


@pytest.mark.parametrize("case", ["keys0", "keys31", "gamma_near_1"])
def test_state_copy_and_perturbation(sb, O, train_series, case):
    """replaced d: get_state(d) after == get_state(s) before (floats and opt), get_hparams(d) == RN32(hp_s × f) with the clamp.
    Every learner: best slot, best_score / best_run and replay memory unchanged; kept learners: state and hyper-parameters too."""
    P, sizes, frac, seed, rnd = 8, [5, 3], 0.5, 11, 4
    keys = {"keys0": (), "keys31": HP, "gamma_near_1": ("gamma", "tau")}[case]
    factors = (0.8, 1.25)
    le, mems = _trained(sb, train_series, P, batch=32, **SMALL)
    if case == "gamma_near_1":
        for l in range(P):
            le.select(l).set_hparams(gamma=0.999, tau=0.9)
        le.select(0)
    before, best0 = _all(le, mems)
    score = np.array([0.3, np.nan, 1.2, -4.0, 0.3, 2.0, -np.inf, 0.5])
    parent = le.exploit(torch.as_tensor(score, device="cuda"), frac, factors=factors, keys=keys, seed=seed, round=rnd, groups=sizes)
    parent = parent.cpu().numpy()
    want, w1 = _restate(O, score, sizes, frac, seed, rnd)
    np.testing.assert_array_equal(parent, want)
    assert (parent >= 0).sum() == 2 + 1
    after, best1 = _all(le, mems)
    clamped = 0                                          # replaced learners whose γ went through the clamp
    for d in range(P):
        s = parent[d]
        if s >= 0:
            _same(after[d], before[s], (d, s))
            hp = _perturbed(before[s]["hp"], keys, w1[d], factors)
            assert after[d]["hp"] == hp, (d, after[d]["hp"], hp)
            clamped += int(case == "gamma_near_1" and (int(w1[d]) >> 2) & 1 == 1)
        else:
            _same(after[d], before[d], d)
            assert after[d]["hp"] == before[d]["hp"]
        for (wa, ba), (wb, bb) in zip(after[d]["best"], before[d]["best"]):
            np.testing.assert_array_equal(wa, wb)
            np.testing.assert_array_equal(ba, bb)
        for xa, xb in zip(after[d]["mem"], before[d]["mem"]):
            np.testing.assert_array_equal(xa, xb)
    np.testing.assert_array_equal(best0[0], best1[0])
    np.testing.assert_array_equal(best0[1], best1[1])
    if case == "gamma_near_1":
        assert clamped > 0 and all(after[d]["hp"]["gamma"] <= 1.0 and after[d]["hp"]["tau"] <= 1.0 for d in range(P))


@pytest.mark.parametrize("tc", [0, 1])
def test_twin_trains_identically(sb, train_series, tc):
    """after an exploit, K Philox-minibatch updates equal those of a twin population that received the post-exploit states through
    set_state / set_hparams: nets, ADAM state and losses, on the tiled fp32 path and on tensor cores (B = 256)."""
    P, B = 6, (256 if tc else 64)
    kw = dict(batch=B, use_tensor_cores=tc, **SMALL)
    le, mems = _trained(sb, train_series, P, seed=90, **kw)
    score = torch.as_tensor(np.array([1.0, -2.0, 3.0, 0.5, -1.0, 2.5]), device="cuda")
    parent = le.exploit(score, 0.5, keys=HP, seed=4, round=2).cpu().numpy()
    assert (parent >= 0).sum() == 3
    post, _ = _all(le)
    twin = _population(sb, mems, **kw)
    twin.init(1234)
    for l in range(P):
        twin.select(l).set_state(post[l]["state"], post[l]["opt"])
        twin.set_hparams(**post[l]["hp"])
    twin.select(0)
    for x in (le, twin):
        x.replay(mems, rng_rpl=77, n_updates=4)
    a, _ = _all(le)
    b, _ = _all(twin)
    for l in range(P):
        _same(a[l], b[l], l)
        assert a[l]["hp"] == b[l]["hp"]
        assert le.select(l).losses() == twin.select(l).losses(), l
    # the updates moved the replaced learners away from the copied states
    d = int(np.flatnonzero(parent >= 0)[0])
    assert a[d]["state"].tobytes() != post[d]["state"].tobytes()


def test_get_hparams_mirror_and_later_set(sb, O, train_series):
    """get_hparams after an exploit shows the device values; a ddpg_set_hparams enqueued after the exploit (no synchronisation in
    between) wins for its learner."""
    P = 4
    le, mems = _trained(sb, train_series, P, batch=32, **SMALL)
    before, _ = _all(le)
    score = torch.as_tensor(np.array([3.0, 2.0, 1.0, 0.0]), device="cuda")
    parent = le.exploit(score, 0.5, factors=(0.5, 2.0), keys=HP, seed=8, round=0)
    lib = sb._lib.lib()
    le.select(3)
    assert lib.ddpg_set_hparams(le._h, 1e-4, 2e-4, 0.5, 0.25, 3.0) == 0      # enqueued behind the exploit
    parent = parent.cpu().numpy()
    np.testing.assert_array_equal(parent, [-1, -1, parent[2], parent[3]])
    assert parent[2] in (0, 1) and parent[3] in (0, 1)
    got = {l: le.select(l).get_hparams() for l in range(P)}
    assert got[3] == dict(lr_actor=np.float32(1e-4).item(), lr_critic=np.float32(2e-4).item(), gamma=0.5, tau=0.25, noise_scale=3.0)
    want, w1 = _restate(O, score.cpu().numpy(), [P], 0.5, 8, 0)
    np.testing.assert_array_equal(parent, want)
    assert got[2] == _perturbed(before[parent[2]]["hp"], HP, w1[2], (0.5, 2.0)) != before[parent[2]]["hp"]
    assert got[0] == before[0]["hp"] and got[1] == before[1]["hp"]


def test_invalid_arguments_launch_nothing(sb, train_series):
    L = sb._lib
    lib = L.lib()
    P = 4
    le, mems = _trained(sb, train_series, P, batch=32, **SMALL)
    before, _ = _all(le)
    score = torch.as_tensor(np.array([3.0, 2.0, 1.0, 0.0]), device="cuda")
    parent = torch.full((P,), 7, dtype=torch.int32, device="cuda")
    sp, pp = C.c_void_p(score.data_ptr()), C.c_void_p(parent.data_ptr())

    def params(**kw):
        p = L.DdpgExploitParams()
        p.frac, p.factor_lo, p.factor_hi, p.keys, p.round, p.seed, p.n_groups = 0.5, 0.8, 1.25, 31, 0, 1, 0
        for k, v in kw.items():
            if k == "group_start":
                p.group_start[:len(v)] = v
            else:
                setattr(p, k, v)
        return p

    assert lib.ddpg_exploit(None, sp, C.byref(params()), pp) == L.ERR_INVALID
    assert lib.ddpg_exploit(le._h, None, C.byref(params()), pp) == L.ERR_INVALID
    assert lib.ddpg_exploit(le._h, sp, None, pp) == L.ERR_INVALID
    bad = [dict(frac=float("nan")), dict(frac=-0.1), dict(frac=0.51), dict(factor_lo=0.0), dict(factor_hi=-1.0), dict(factor_lo=float("inf")),
           dict(factor_hi=float("nan")), dict(keys=-1), dict(keys=32), dict(n_groups=-1), dict(n_groups=17),
           dict(n_groups=2, group_start=[1, 2, P]), dict(n_groups=2, group_start=[0, 2, P - 1]), dict(n_groups=3, group_start=[0, 2, 2, P]),
           dict(n_groups=2, group_start=[0, 3, 2])]
    for kw in bad:
        assert lib.ddpg_exploit(le._h, sp, C.byref(params(**kw)), pp) == L.ERR_INVALID, kw
    torch.cuda.synchronize()
    assert bool((parent == 7).all())
    after, _ = _all(le)
    for l in range(P):
        _same(before[l], after[l], l)
        assert before[l]["hp"] == after[l]["hp"]
    assert lib.ddpg_exploit(le._h, sp, C.byref(params(n_groups=2, group_start=[0, 2, P])), pp) == L.OK
    np.testing.assert_array_equal(parent.cpu().numpy(), [-1, 0, -1, 2])
    one = sb.Learner(params=sb.default_ddpg_params(batch=32, **SMALL))
    one.init(1)
    st0 = one.get_state()
    p1 = one.exploit(torch.zeros(1, dtype=torch.float64, device="cuda"), 0.5, seed=1)
    assert p1.cpu().numpy().tolist() == [-1]
    np.testing.assert_array_equal(one.get_state()[0], st0[0])


def _driver(sb, train_series, eval_series):
    drv = sb.PopulationDriver(train_series, chargers=[98, 98, 98, 98, 4, 4, 4], seeds=[11, 12, 13, 14, 15, 16, 17], n_envs=8, mem_size=8 * 72,
                              eval_series=eval_series, test_runs=5, batch=64, use_tensor_cores=0, **SMALL)
    return drv


def _extend(st, E, P):
    st = copy.deepcopy(st)
    n = E - len(st["total_reward"])
    st["total_reward"] = np.concatenate([st["total_reward"], np.zeros((n, P))])
    st["score_mean"] = np.concatenate([st["score_mean"], np.zeros((n, P))])
    st["parent"] = np.concatenate([st["parent"], np.full((n, P), -1, np.int32)])
    st["hparams"] = np.concatenate([st["hparams"], np.zeros((n, P, 5), np.float32)])
    return st


def test_driver_pbt_groups_and_resume(sb, O, train_series, tmp_path):
    """run_episodes(pbt=...) on two charger runs (4 + 3 learners), test_every = 1: every parent is the restated choice inside its
    charger run; interrupted after 2 episodes, checkpointed, reloaded into a fresh driver and continued, the run ends bit-identical
    to the uninterrupted one (states, hyper-parameters, lineage, scores)."""
    P, E = 7, 4
    ev_ser = sb.series.synth_charger98(1440, seed=31)
    pbt = dict(every=1, frac=0.5, factors=(0.8, 1.25), keys=("lr_actor", "lr_critic", "noise_scale"), seed=5)
    full = _driver(sb, train_series, ev_ser)
    full.populate_memory()
    full.min_max_buffer()
    st = full.run_episodes(E, test_every=1, pbt=pbt)
    assert st["parent"].shape == (E, P) and st["hparams"].shape == (E, P, 5)
    for r in range(E):
        want, _ = _restate(O, st["score_mean"][r], [4, 3], 0.5, 5, r)
        np.testing.assert_array_equal(st["parent"][r], want, err_msg=str(r))
        for d, s in enumerate(st["parent"][r]):
            assert s < 0 or (d < 4) == (s < 4), (r, d, s)     # never across chargers
    assert (st["parent"] >= 0).sum() == E * (2 + 1)
    for l in range(P):
        hp = full.learner.select(l).get_hparams()
        np.testing.assert_array_equal(st["hparams"][-1, l], np.array([hp[k] for k in HP], np.float32))
    # interrupted after episode 2, checkpointed with the scores, resumed in a fresh driver
    part = _driver(sb, train_series, ev_ser)
    part.populate_memory()
    part.min_max_buffer()
    st2 = part.run_episodes(2, test_every=1, pbt=pbt)
    path = str(tmp_path / "pbt.npz")
    sb.tracker.save_checkpoint(path, part.learner, memories=part.mems, **st2)
    fresh = _driver(sb, train_series, ev_ser)
    z = sb.tracker.load_checkpoint(path, fresh.learner, memories=fresh.mems)
    st3 = {k: np.array(z[k]) for k in ("total_reward", "score_mean", "best_run", "best_score", "parent", "hparams")}
    st3 = fresh.run_episodes(E, test_every=1, start_ep=3, state=_extend(st3, E, P), pbt=pbt)
    for k in ("total_reward", "score_mean", "best_run", "best_score", "parent", "hparams"):
        np.testing.assert_array_equal(st3[k], st[k], err_msg=k)
    a, _ = _all(full.learner)
    b, _ = _all(fresh.learner)
    for l in range(P):
        _same(a[l], b[l], l)
        assert a[l]["hp"] == b[l]["hp"]
