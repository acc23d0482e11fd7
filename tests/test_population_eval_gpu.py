"""Evaluation, best-actor bookkeeping and inference for every learner of a population (ddpg_evaluate, ddpg_keep_best,
PopulationDriver.run_episodes / inference): run_episodes of DDPG.jl:244-298 and the driver's inference (DDPG_reinforce_charger_v1.jl:87-105).
Everything is compared bit for bit: a learner evaluated inside a population must get exactly what it gets on a one-learner handle."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SMALL = dict(batch=64, l1=48, l2=64, use_tensor_cores=0)


def _actor(le, net=0):
    return [le.get_layer(net, k) for k in range(3)]


def _same_layers(a, b):
    for (wa, ba), (wb, bb) in zip(a, b):
        np.testing.assert_array_equal(wa, wb)
        np.testing.assert_array_equal(ba, bb)


def _mean_in_order(x):
    s = 0.0
    for v in x:
        s += float(v)
    return s / len(x)


def _norm_of(le):
    st, _ = le.get_state()
    return st[-18:-9].copy(), st[-9:].copy()


@pytest.mark.parametrize("two_groups", [False, True])
def test_evaluate_one_learner_equals_rollout(sb, train_series, two_groups):
    """ddpg_evaluate(ACTOR) on a one-learner handle is ddpg_rollout(sigma = 0): returns, traces, actions, final state and idx."""
    le = sb.Learner()
    le.init(21)
    le.set_norm(np.zeros(9, np.float32), np.linspace(1, 9, 9).astype(np.float32))
    kw = dict(groups=[(98, 5), (4, 8)]) if two_groups else dict(n_envs=13)
    envs = [sb.Shems(72, train_series, env_id_base=40, **kw) for _ in range(2)]
    outs = []
    for env, ev in zip(envs, (False, True)):
        env.reset(rng=9)
        if ev:
            o = le.evaluate(env, 72, want_trace=True, want_actions=True)
        else:
            o = le.rollout(env, 72, sigma=0.0, rng_ep=5, want_trace=True, want_actions=True)
        torch.cuda.synchronize()
        outs.append((o, env.state, env.idx))
    (a, sa, ia), (b, sb_, ib) = outs
    for k in ("ep_return", "trace", "actions"):
        assert torch.equal(a[k], b[k]), k
    np.testing.assert_array_equal(sa, sb_)
    np.testing.assert_array_equal(ia, ib)
    assert float(a["ep_return"].abs().sum()) > 0


@pytest.mark.parametrize("n", [1, 5, 13])
def test_population_evaluate_equals_one_learner_handles(sb, train_series, n):
    """P = 4 learners with their own weights and s_min / s_max, two charger groups with different series: every learner's slice
    equals a one-learner handle holding that learner's actor and norm on an env of its n instances."""
    P, T, E = 4, 72, 1000
    ser2 = np.stack([train_series, sb.series.synth_charger98(train_series.shape[1], seed=7)])
    chargers = [98, 98, 4, 4]
    pop = sb.Learner(params=sb.default_ddpg_params(population=P))
    pop.init(5)
    rng = np.random.default_rng(n)
    for l in range(P):
        pop.select(l).set_norm(rng.uniform(-1, 0, 9).astype(np.float32), rng.uniform(2, 9, 9).astype(np.float32))
    env = sb.Shems(T, ser2, groups=[(98, 2 * n), (4, 2 * n)], env_id_base=E)
    env.reset(rng=17)
    obs0, idx0 = env.state, env.idx
    for best in (False, True):
        if best:   # the best-actor slots: give them other weights than the actors (learner l: the actor of learner P-1-l)
            acts = [_actor(pop.select(l)) for l in range(P)]
            for l in range(P):
                for k, (w, b) in enumerate(acts[P - 1 - l]):
                    pop.select(l).set_layer(sb._lib.NET_ACTOR_BEST, k, w, b)
            env.set_state(obs0, idx0)
        out = pop.evaluate(env, T, best=best, want_trace=True, want_actions=True)
        torch.cuda.synchronize()
        obs1, idx1 = env.state, env.idx
        for l in range(P):
            one = sb.Learner()
            for k, (w, b) in enumerate(_actor(pop.select(l), sb._lib.NET_ACTOR_BEST if best else sb._lib.NET_ACTOR)):
                one.set_layer(0, k, w, b)
            one.set_norm(*_norm_of(pop.select(l)))
            g = l // 2
            e1 = sb.Shems(T, ser2[g], n_envs=n, charger_id=chargers[l], env_id_base=E + l * n)
            sl = slice(l * n, (l + 1) * n)
            e1.set_state(obs0[:, sl], idx0[sl])
            o1 = one.evaluate(e1, T, want_trace=True, want_actions=True)
            torch.cuda.synchronize()
            assert torch.equal(out["ep_return"][sl], o1["ep_return"]), (best, l)
            assert torch.equal(out["trace"][:, :, sl], o1["trace"]), (best, l)
            assert torch.equal(out["actions"][:, :, sl], o1["actions"]), (best, l)
            np.testing.assert_array_equal(obs1[:, sl], e1.state)
            np.testing.assert_array_equal(idx1[sl], e1.idx)
    r = out["ep_return"].view(P, n)
    assert not torch.equal(r[0], r[1])


def test_keep_best_follows_the_strict_rule(sb):
    """ddpg_keep_best on scripted returns: best_score / best_run follow score > best (a tie and a NaN never win), the ACTOR_BEST slot
    holds the actor of the winning call, the other learners are untouched, score_dev is the index-order Float64 mean."""
    P, n = 4, 5
    le = sb.Learner(params=sb.default_ddpg_params(population=P, **SMALL))
    rng = np.random.default_rng(3)
    base = rng.normal(0, 1, (P, n))
    # target scores per call (learner 3 never wins: NaN, then below the -100000 start, then NaN)
    script = [[-5.0, np.nan, -200000.0, np.nan], [-5.0, -7.0, -3.0, -300000.0], [-4.0, np.nan, -3.0, np.nan]]
    snaps, want_score, want_run, want_actor = [], np.full(P, -100000.0), np.zeros(P, np.int32), [None] * P
    first = None
    for call, targets in enumerate(script, start=1):
        le.init(100 + call)                                   # a different actor at every call
        snaps.append([_actor(le.select(l)) for l in range(P)])
        ret = np.empty((P, n))
        for l, t in enumerate(targets):
            ret[l] = base[l] + t if not np.isnan(t) else np.where(np.arange(n) == 2, np.nan, base[l])
        if call == 1:
            first = ret.copy()
        if call == 2:
            ret[0] = first[0]                                 # learner 0: exactly the score of call 1 (a tie)
        sc = le.keep_best(torch.as_tensor(ret.ravel(), device="cuda"), n, call).cpu().numpy()
        for l in range(P):
            m = _mean_in_order(ret[l])
            assert (np.isnan(m) and np.isnan(sc[l])) or sc[l] == m, (call, l)
            if m > want_score[l]:
                want_score[l], want_run[l], want_actor[l] = m, call, snaps[-1][l]
    got_score, got_run = le.best()
    np.testing.assert_array_equal(got_run, [3, 2, 2, 0])
    np.testing.assert_array_equal(got_run, want_run)
    np.testing.assert_array_equal(got_score, want_score)
    for l in range(P):
        best = _actor(le.select(l), sb._lib.NET_ACTOR_BEST)
        if want_actor[l] is None:
            assert all((w == 0).all() and (b == 0).all() for w, b in best)
        else:
            _same_layers(best, want_actor[l])
    le.set_best([1.0, 2.0, 3.0, 4.0], [5, 6, 7, 8])
    s, r = le.best()
    np.testing.assert_array_equal(s, [1.0, 2.0, 3.0, 4.0])
    np.testing.assert_array_equal(r, [5, 6, 7, 8])


def _driver(sb, train_series, eval_series, **kw):
    drv = sb.PopulationDriver(train_series, chargers=[98, 98, 4], seeds=[11, 12, 13], n_envs=8, mem_size=8 * 72, eval_series=eval_series,
                              test_runs=5, **SMALL, **kw)
    drv.populate_memory()
    drv.min_max_buffer()
    return drv


def test_run_episodes_best_actor_and_inference(sb, train_series, tmp_path):
    """PopulationDriver.run_episodes (P = 3, test_every = 1): re-evaluating a best actor reproduces its score_mean entry, every
    score_mean entry is what the learner's actor scores on a one-learner handle with its own evaluation env, best_run is the first argmax, inference(best=True) equals a one-learner Driver.inference with that actor; a checkpoint round trip followed
    by more episodes equals carrying on without one."""
    P, E = 3, 4
    ev_ser = sb.series.synth_charger98(1440, seed=31)
    te_ser = sb.series.synth_charger98(300, seed=32)
    drv = _driver(sb, train_series, ev_ser)
    calls = []
    st = drv.run_episodes(2, test_every=1, on_best=lambda l, i, s: calls.append((l, i, s)))
    path = str(tmp_path / "pop.npz")
    sb.tracker.save_checkpoint(path, drv.learner, memories=drv.mems)
    st2 = copy.deepcopy(st)
    st2["total_reward"] = np.concatenate([st2["total_reward"], np.zeros((E - 2, P))])
    st2["score_mean"] = np.concatenate([st2["score_mean"], np.zeros((E - 2, P))])
    st = drv.run_episodes(E, test_every=1, start_ep=3, state=copy.deepcopy(st2))
    assert st["score_mean"].shape == (E, P) and st["total_reward"].shape == (E, P)
    for l in range(P):
        i = int(np.argmax(st["score_mean"][:, l]))
        assert st["best_run"][l] == i + 1 and st["best_score"][l] == st["score_mean"][i, l]
    s_dev, r_dev = drv.learner.best()
    np.testing.assert_array_equal(s_dev, st["best_score"])
    np.testing.assert_array_equal(r_dev, st["best_run"])
    assert [(l, i) for l, i, _ in calls][:P] == [(0, 1), (1, 1), (2, 1)]
    # re-evaluate every best actor: the same round reproduces score_mean[best_run][l] exactly
    ret = drv.learner.evaluate(drv.reset_eval(123 * 1000 + 1), 72, best=True)["ep_return"].view(P, 5).cpu().numpy()
    for l in range(P):
        assert _mean_in_order(ret[l]) == st["score_mean"][st["best_run"][l] - 1, l]
    # every learner is scored on the starts a one-learner run sees: its actor (the last round) and its best actor (round best_run),
    # with its norm, on a one-learner handle and an eval env of test_runs instances (env_id_base 0) reset with the same rng
    for l in range(P):
        for net, row in ((sb._lib.NET_ACTOR, E - 1), (sb._lib.NET_ACTOR_BEST, st["best_run"][l] - 1)):
            one = sb.Learner(params=sb.default_ddpg_params(**SMALL))
            for k, (w, b) in enumerate(_actor(drv.learner.select(l), net)):
                one.set_layer(0, k, w, b)
            one.set_norm(*_norm_of(drv.learner.select(l)))
            env1 = sb.Shems(1439, ev_ser, n_envs=5, charger_id=drv.chargers[l])
            env1.reset(rng=123 * 1000 + 1)
            r1 = one.evaluate(env1, 72)["ep_return"].cpu().numpy()
            assert _mean_in_order(r1) == st["score_mean"][row, l], (l, net)
    # inference with the best actors vs one-learner Driver.inference
    rets, trace = drv.inference(te_ser)
    assert trace.shape == (299, 23, P)
    for l in range(P):
        le = sb.Learner(params=sb.default_ddpg_params(**SMALL))
        for k, (w, b) in enumerate(_actor(drv.learner.select(l), sb._lib.NET_ACTOR_BEST)):
            le.set_layer(0, k, w, b)
        le.set_norm(*_norm_of(drv.learner.select(l)))
        env1 = sb.Shems(299, te_ser, n_envs=1, charger_id=drv.chargers[l])
        d1 = sb.Driver(env1, learner=le, mem_size=72)
        r1, tr1 = d1.inference(env1, 299)
        assert torch.equal(rets[l:l + 1], r1) and torch.equal(trace[:, :, l:l + 1], tr1), l
    sums = sb.tracker.write_population_results(str(tmp_path / "inf"), trace, drv.chargers, drv.seeds, st["best_run"], st["best_score"])
    lines = open(tmp_path / "inf" / "results_summary.csv").read().splitlines()
    assert len(lines) == P + 1 and lines[0].split(",") == sb.tracker.SUMMARY_HEADER
    assert sums[1]["rewards"] == pytest.approx(float(rets[1]), rel=1e-12)
    # resume from the checkpoint written after episode 2 in a fresh driver
    drv2 = sb.PopulationDriver(train_series, chargers=[98, 98, 4], seeds=[11, 12, 13], n_envs=8, mem_size=8 * 72, eval_series=ev_ser, test_runs=5,
                               **SMALL)
    sb.tracker.load_checkpoint(path, drv2.learner, memories=drv2.mems)
    st3 = drv2.run_episodes(E, test_every=1, start_ep=3, state=copy.deepcopy(st2))
    for k in ("total_reward", "score_mean", "best_run", "best_score"):
        np.testing.assert_array_equal(st3[k], st[k], err_msg=k)
    for l in range(P):
        _same_layers(_actor(drv2.learner.select(l), sb._lib.NET_ACTOR_BEST), _actor(drv.learner.select(l), sb._lib.NET_ACTOR_BEST))
        _same_layers(_actor(drv2.learner.select(l)), _actor(drv.learner.select(l)))
    # a fresh run_episodes starts from zero best actors, not from what an earlier call on the handle kept
    st0 = drv.run_episodes(0, test_every=1)
    assert st0["score_mean"].shape == (0, P) and (drv.learner.best()[1] == 0).all()
    for l in range(P):
        assert all((w == 0).all() and (b == 0).all() for w, b in _actor(drv.learner.select(l), sb._lib.NET_ACTOR_BEST))


def test_evaluate_errors_launch_nothing(sb, train_series):
    """the status codes of ddpg_evaluate, with the output buffer left as it was; ACTOR_BEST where a call does not take it."""
    L = sb._lib
    lib = L.lib()
    pop = sb.Learner(params=sb.default_ddpg_params(population=2, **SMALL))
    pop.init(1)
    env = sb.Shems(72, train_series, n_envs=8)
    ret = torch.full((8,), 7.0, dtype=torch.float64, device="cuda")

    def call(le, e, net=L.NET_ACTOR, T=72):
        return lib.ddpg_evaluate(le._h, e._h, net, T, 0, C.c_void_p(ret.data_ptr()), None, None)

    assert call(pop, env) == L.ERR_STATE                                            # reset! first
    env.reset(rng=1)
    assert call(pop, env, T=4400) == L.ERR_BOUNDS                                   # leaves the series
    assert call(pop, env, net=L.NET_CRITIC) == L.ERR_INVALID
    assert call(pop, env, T=0) == L.ERR_INVALID
    split = sb.Shems(72, train_series, groups=[(98, 3), (4, 5)])                    # a group boundary inside learner 0's 4 instances
    split.reset(rng=1)
    assert call(pop, split) == L.ERR_INVALID
    wide = sb.Learner(params=sb.default_ddpg_params(population=2, batch=64, l1=300, l2=64))
    assert call(wide, env) == L.ERR_INVALID                                         # outside the cluster kernel's plan
    odd = sb.Shems(72, train_series, n_envs=7)
    odd.reset(rng=1)
    assert call(pop, odd) == L.ERR_INVALID                                          # 7 instances do not split over 2 learners
    torch.cuda.synchronize()
    assert bool((ret == 7.0).all())
    assert lib.ddpg_get_grad(pop._h, L.NET_ACTOR_BEST, 0, None, None) == L.ERR_INVALID
    assert lib.ddpg_num_params(pop._h, L.NET_ACTOR_BEST) == lib.ddpg_num_params(pop._h, L.NET_ACTOR)
    assert lib.ddpg_num_params(pop._h, 5) == 0
    assert lib.ddpg_keep_best(pop._h, None, 4, 1, None) == L.ERR_INVALID
    assert call(pop, env) == L.OK
