"""Per-learner hyper-parameters (ddpg_set_hparams / ddpg_get_hparams): η_act, η_crit, γ, τ and the exploration-noise scale.

A learner whose values were set after ddpg_create must compute exactly what a learner created with those values computes: the
compared handles issue identical launches, so "equal" is equal bits.  Noise uses σ_eff = float32(σ × noise_scale)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

P = 4
SMALL = dict(l1=48, l2=64)
TUPLES = [dict(lr_actor=1e-4, lr_critic=1e-3, gamma=0.99, tau=1e-3), dict(lr_actor=3e-4, lr_critic=5e-4, gamma=0.95, tau=5e-3),
          dict(lr_actor=5e-5, lr_critic=2e-3, gamma=0.9, tau=1e-2), dict(lr_actor=2e-4, lr_critic=1e-3, gamma=0.8, tau=2e-3)]
SCALES = [0.05, 0.1, 0.2, 0.3]


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


def _snapshot(le, l):
    le.select(l)
    st, opt = le.get_state()
    return st, opt, np.array(le.losses(), np.float32)


def _assert_same(a, b, what=""):
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y, err_msg=what)


@pytest.mark.parametrize("tc", [0, 1])
def test_mixed_population_equals_homogeneous_twins(sb, train_series, tc):
    """Learner l of a population with four distinct (η_a, η_c, γ, τ) equals learner l of a population whose DdpgParams carry its values,
    after updates from host indices and then from Philox draws.  tc = 1 at B = 256 takes the tensor-core path with the forward-chain
    kernels (TD target in their epilogue) and the fp32 ADAM; tc = 0 the tiled GEMMs (TD target in the skinny epilogue)."""
    B = 256 if tc else 64
    mems = [_memory(sb, train_series, seed=30 + l) for l in range(P)]
    idx = np.stack([np.random.default_rng(l).integers(0, len(mems[l]), (3, B)) for l in range(P)]).astype(np.int32)

    def run(le):
        le.replay(mems, n_updates=3, idx=idx)
        le.replay(mems, rng_rpl=77, n_updates=4)
        return le

    mixed = _population(sb, mems, batch=B, use_tensor_cores=tc, **SMALL)
    for l, t in enumerate(TUPLES):
        mixed.select(l).set_hparams(**t)
    run(mixed)
    for l, t in enumerate(TUPLES):
        twin = run(_population(sb, mems, batch=B, use_tensor_cores=tc, **SMALL, **t))
        _assert_same(_snapshot(mixed, l), _snapshot(twin, l), "learner %d" % l)
        twin.close()
    # the learners really differ: learner 1 of the mixed population is not learner 1 of a default population
    default = run(_population(sb, mems, batch=B, use_tensor_cores=tc, **SMALL))
    assert _snapshot(mixed, 1)[0].tobytes() != _snapshot(default, 1)[0].tobytes()


def test_noise_scale_in_act_and_act_ou(sb, train_series):
    """σ = 1 with per-learner scales equals the default population called with σ = scale (Gaussian SoA act, OU with Philox and with
    injected z)."""
    n = 40
    mems = [_memory(sb, train_series, seed=40 + l) for l in range(P)]
    mixed, twin = _population(sb, mems, **SMALL), _population(sb, mems, **SMALL)
    for l, s in enumerate(SCALES):
        mixed.select(l).set_hparams(noise_scale=s)
    mixed.select(0)
    rng = np.random.default_rng(5)
    obs = torch.as_tensor(rng.uniform(0, 1, (9, P * n)).astype(np.float32), device="cuda")
    a_m, sc_m = mixed.act(obs, sigma=1.0, rng_act=11, step=3, soa=True)
    for l, s in enumerate(SCALES):
        a_t, sc_t = twin.act(obs, sigma=s, rng_act=11, step=3, soa=True)
        sl = slice(l * n, (l + 1) * n)
        assert torch.equal(a_m[:, sl], a_t[:, sl]) and torch.equal(sc_m[:, sl], sc_t[:, sl]), l
    obs_p = obs.view(9, P, n).permute(1, 0, 2).contiguous()
    x0 = torch.as_tensor(rng.normal(0, 0.3, (P, 2, n)).astype(np.float32), device="cuda")
    z = torch.as_tensor(rng.normal(0, 1, (P, 2, n)), device="cuda")
    for zz in (None, z):
        xm = x0.clone()
        a_m, sc_m = mixed.act_ou(obs_p, xm, sigma=1.0, rng_act=12, step=4, z=zz)
        for l, s in enumerate(SCALES):
            xt = x0.clone()
            a_t, sc_t = twin.act_ou(obs_p, xt, sigma=s, rng_act=12, step=4, z=zz)
            assert torch.equal(a_m[l], a_t[l]) and torch.equal(sc_m[l], sc_t[l]) and torch.equal(xm[l], xt[l]), l


@pytest.mark.parametrize("kind", ["gn", "ou"])
def test_noise_scale_in_training_episode(sb, train_series, kind):
    """One native training ddpg_episode on a population with σ = 1 and per-learner scales: learner l's returns, noise_eps and
    weights equal those of learner l of a default population trained with σ = its scale."""
    n, T = 8, 12

    def episode(le, sigma):
        mems = [_memory(sb, train_series, seed=50 + l, capacity=4096) for l in range(P)]
        for l, m in enumerate(mems):
            le.select(l).set_norm(*m.min_max_buffer(len(m), rng_mm=l))
        le.select(0)
        le.set_noise(kind)
        env = sb.Shems(72, train_series, n_envs=P * n)
        env.reset(rng=9)
        ret, nz = le.episode(env, mems, T, train=True, sigma=sigma, rng_ep=31, updates_per_step=1, want_noise=True)
        return ret.cpu().numpy(), nz.cpu().numpy()

    mixed = _population(sb, [_memory(sb, train_series, seed=50 + l) for l in range(P)], batch=32, **SMALL)
    for l, s in enumerate(SCALES):
        mixed.select(l).set_hparams(noise_scale=s)
    ret_m, nz_m = episode(mixed, 1.0)
    for l, s in enumerate(SCALES):
        twin = _population(sb, [_memory(sb, train_series, seed=50 + k) for k in range(P)], batch=32, **SMALL)
        ret_t, nz_t = episode(twin, s)
        sl = slice(l * n, (l + 1) * n)
        np.testing.assert_array_equal(ret_m[sl], ret_t[sl])
        np.testing.assert_array_equal(nz_m[sl], nz_t[sl])
        np.testing.assert_array_equal(_snapshot(mixed, l)[0], _snapshot(twin, l)[0])
        twin.close()
    assert np.any(nz_m[:n] != nz_m[n:2 * n])


X = dict(lr_actor=3e-4, lr_critic=5e-4, gamma=0.9, tau=4e-3)


@pytest.mark.parametrize("path", ["fused", "tiled", "wide"])
def test_single_learner_set_equals_created(sb, train_series, path):
    """P = 1: a default handle plus set_hparams(X) equals a handle created with X — updates on the cluster-fused path, on the tiled
    path (ddpg_set_fused(0)), and ddpg_rollout with σ > 0 on the persistent cluster kernel and (l2 = 640) on the act + step!
    launch pair.  noise_scale s with σ equals σ_eff = float32(σ s) in act() and in both rollout paths."""
    widths = dict(l1=64, l2=640) if path == "wide" else dict(l1=64, l2=128)
    mem = _memory(sb, train_series, n=32)
    norm = mem.min_max_buffer(len(mem), rng_mm=1)

    def make(**kw):
        le = sb.Learner(params=sb.default_ddpg_params(batch=64, **widths, **kw))
        le.set_fused(path == "fused")
        le.init(3)
        le.set_norm(*norm)
        return le
    a, b = make(), make(**X)
    a.set_hparams(**X)
    for le in (a, b):
        le.replay(mem, rng_rpl=5, n_updates=6)
    _assert_same(_snapshot(a, 0), _snapshot(b, 0))

    def rollout(le, sigma):
        env = sb.Shems(72, train_series, n_envs=20)
        env.reset(rng=4)
        out = le.rollout(env, 24, sigma=sigma, rng_ep=8, want_actions=True)
        return out["ep_return"].cpu().numpy(), out["actions"].cpu().numpy()
    _assert_same(rollout(a, 0.3), rollout(b, 0.3))
    sig, s = 0.3, 0.7
    eff = float(np.float32(sig) * np.float32(s))
    a.set_hparams(noise_scale=s)
    assert a.get_hparams()["noise_scale"] == np.float32(s)
    ra, rb = rollout(a, sig), rollout(b, eff)
    _assert_same(ra, rb)
    assert not np.array_equal(ra[1], rollout(b, sig)[1])
    obs = torch.as_tensor(np.random.default_rng(2).uniform(0, 1, (9, 16)).astype(np.float32), device="cuda")
    for x, y in zip(a.act(obs, sigma=sig, rng_act=3, step=2), b.act(obs, sigma=eff, rng_act=3, step=2)):
        assert torch.equal(x, y)


@pytest.mark.parametrize("cfg", [dict(P=1, fused=True, tc=0, B=64), dict(P=1, fused=False, tc=0, B=64), dict(P=4, fused=False, tc=1, B=256)])
def test_change_mid_run_without_recapture(sb, train_series, cfg):
    """A runs K updates with X, set_hparams(Y), K more (its captured update graph is replayed, not re-captured); B is created with Y,
    takes A's state after the first K updates and runs K updates.  A must equal B: no stale by-value η, γ, τ in the graph."""
    Y = dict(lr_actor=5e-5, lr_critic=2e-3, gamma=0.8, tau=1e-2)
    pop = cfg["P"]
    mems = [_memory(sb, train_series, seed=60 + l) for l in range(pop)]

    def make(**kw):
        le = _population(sb, mems, batch=cfg["B"], use_tensor_cores=cfg["tc"], **SMALL, **kw)
        le.set_fused(cfg["fused"])
        return le

    def replay(le, r):
        le.replay(mems if pop > 1 else mems[0], rng_rpl=r, n_updates=3)
    a, b = make(**X), make(**Y)
    replay(a, 1)
    mid = [a.select(l).get_state() for l in range(pop)]
    for l in range(pop):
        a.select(l).set_hparams(**Y)
        b.select(l).set_state(*mid[l])
    replay(a, 2)
    replay(b, 2)
    for l in range(pop):
        _assert_same(_snapshot(a, l), _snapshot(b, l), "learner %d" % l)


def test_validation_and_checkpoint(sb, train_series, tmp_path):
    mems = [_memory(sb, train_series, seed=70 + l) for l in range(P)]
    le = _population(sb, mems, batch=32, **SMALL)
    for l, t in enumerate(TUPLES):
        le.select(l).set_hparams(**t, noise_scale=SCALES[l])
    le.select(2)
    before = le.get_hparams()
    assert before == {k: float(np.float32(v)) for k, v in dict(TUPLES[2], noise_scale=SCALES[2]).items()}
    for bad in (dict(lr_actor=float("nan")), dict(lr_critic=-1e-4), dict(gamma=1.5), dict(tau=-0.1), dict(noise_scale=-1.0),
                dict(gamma=float("inf"))):
        with pytest.raises(sb._lib.ShemsError):
            le.set_hparams(**bad)
        assert le.get_hparams() == before
    with pytest.raises(sb._lib.ShemsError):
        le.select(P)
    assert le.get_hparams() == before
    le.set_hparams(gamma=1.0, tau=0.0, lr_actor=0.0, noise_scale=0.0)   # the closed ends of the ranges are valid
    le.set_hparams(**TUPLES[2], noise_scale=SCALES[2])
    le.replay(mems, rng_rpl=3, n_updates=2)
    path = str(tmp_path / "ckpt.npz")
    sb.tracker.save_checkpoint(path, le)
    z = np.load(path)
    np.testing.assert_array_equal(z["l1_hparams"], np.array([TUPLES[1][k] for k in ("lr_actor", "lr_critic", "gamma", "tau")] + [SCALES[1]],
                                                            np.float32))
    le2 = _population(sb, mems, batch=32, **SMALL)
    sb.tracker.load_checkpoint(path, le2)
    for l in range(P):
        assert le2.select(l).get_hparams() == le.select(l).get_hparams()
    le.replay(mems, rng_rpl=4, n_updates=2)
    le2.replay(mems, rng_rpl=4, n_updates=2)
    for l in range(P):
        _assert_same(_snapshot(le, l), _snapshot(le2, l))
    # a checkpoint without the key (written before per-learner values existed) loads as before and leaves them alone
    old = {k: z[k] for k in z.files if not k.endswith("_hparams")}
    np.savez(str(tmp_path / "old.npz"), **old)
    le3 = _population(sb, mems, batch=32, **SMALL)
    sb.tracker.load_checkpoint(str(tmp_path / "old.npz"), le3)
    assert le3.select(1).get_hparams() == le3.select(0).get_hparams()
