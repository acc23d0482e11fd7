"""The reference driver's call sequence (RL-SHEMS/DDPG_reinforce_charger_v1.jl:24-108), walked through the C ABI in the order and
with the argument shapes the Julia shim (julia/DdpgB200.jl, SHEMS_B200_RNG=julia) uses — one instance, every random draw made on the
host and injected — next to the CPU oracle fed the same draws:

    Shems(72, train) / Shems(1439, eval)            input.jl:162-164
    actor, critic, targets (Flux init) -> learner   DDPG.jl:30-46           ddpg_set_layer x 12 (adopted on first use)
    populate_memory(env_train; rng)                 driver :28              reset! host draws + shems_rollout(TAPE, tape_unscaled, replay)
    s_min, s_max = min_max_buffer(MIN_EXP_SIZE)     driver :30              replay_sample(idx_host) -> minimum / maximum -> ddpg_set_norm
    run_episodes(...)                               driver :42              per step: ddpg_act(noise) -> shems_step -> replay_push -> ddpg_update(idx)
        every test_every episodes: evaluation       DDPG.jl:266-279         ddpg_rollout (72 steps, one kernel)
        best score -> saveBSON(actor, path="temp")  DDPG.jl:282-289         ddpg_get_layer (actor)
    saveBSON(actor, ...)                            driver :45              ddpg_get_layer (actor)
    global actor = loaded; inference(track = 1)     driver :93-101          ddpg_set_layer (actor) + ddpg_rollout with the 23-column trace
    inference(track < 0)                            driver :105             shems_rollout(RULE, trace)
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def dev(x):
    return torch.as_tensor(np.ascontiguousarray(x), device="cuda")


def test_reference_driver_call_sequence(sb, O, train_series, charger98_test_series, tmp_path):
    T, B, MEM, NUM_EP, TEST_EVERY, TEST_RUNS = 72, 120, 72 * 12, 3, 2, 3
    rng = np.random.default_rng(7)
    P = O.params_for_charger(98)
    eval_series = sb.series.synth_charger98(1440, seed=7)
    env_train, env_eval = sb.Shems(T, train_series, n_envs=1), sb.Shems(1439, eval_series, n_envs=1)
    ref_train, ref_eval = O.OracleEnv(P, train_series, T, 1), O.OracleEnv(P, eval_series, 1439, 1)
    # --- DDPG.jl:30-46: the Flux nets exist first; the learner adopts them
    le, orc = sb.Learner(), O.OracleDdpg(O.default_ddpg_params())
    orc.init(1231)                                   # stands in for Flux's glorot / w_init draws
    for net in range(4):
        for k in range(3):
            le.set_layer(net, k, *orc.get_layer(net, k))
    memory = sb.Replay(MEM)                          # memory = DeviceMemory(MEM_SIZE)
    S = np.zeros((9, 0), np.float32); A = np.zeros((2, 0), np.float32); R = np.zeros(0, np.float32); S2 = np.zeros((9, 0), np.float32)

    def host_reset(env, ref, maxsteps, nrows, deterministic=False):
        if deterministic:
            env.reset(rng=-1); ref.reset(mode=0)
        else:                                        # the two MersenneTwister(rng) draws of shems_LU1.jl:224-225, made on the host
            idx0 = rng.integers(1, nrows - maxsteps + 1, 1).astype(np.int32)
            socb0 = rng.uniform(0, 6.75, 1).astype(np.float32)
            env.reset(idx0=idx0, socb0=socb0); ref.reset(mode=1, idx0=idx0, socb0=socb0)

    # --- populate_memory (driver :28): random actions drawn on the host, taped, a stored unscaled
    while len(memory) < MEM:
        host_reset(env_train, ref_train, T, train_series.shape[1])
        a = (rng.random((T, 2, 1)) * 2 - 1).astype(np.float32)
        env_train.rollout(sb.POLICY_TAPE, T, tape=dev(a), replay=memory, tape_unscaled=True, want_return=False)
        for t in range(T):
            s = ref_train.obs.copy()
            r, s2, _ = ref_train.step(((a[t].astype(np.float64) + 1) * 0.5).astype(np.float32))
            S = np.concatenate([S, s], 1); A = np.concatenate([A, a[t]], 1); R = np.concatenate([R, r.astype(np.float32)]); S2 = np.concatenate([S2, s2], 1)
    for got, want in zip(memory.get()[:4], (S, A, R, S2)):
        assert got.tobytes() == want.tobytes()       # the device memory holds exactly the reference loop's transitions
    # --- min_max_buffer (driver :30): getData's index draws on the host -> fetch -> minimum/maximum (memory_plotting_saving.jl:50-53)
    idx = rng.integers(0, len(memory), MEM).astype(np.int32)
    s_smp = memory.sample(MEM, idx=idx)[0].cpu().numpy()
    s_min, s_max = s_smp.min(axis=1), s_smp.max(axis=1)
    np.testing.assert_array_equal(s_min, S[:, idx].min(axis=1))
    le.set_norm(s_min, s_max); orc.set_norm(s_min, s_max)
    # --- run_episodes (driver :42)
    total_reward, noise_mean, score_mean = np.zeros(NUM_EP, np.float32), np.zeros(NUM_EP, np.float32), np.zeros(-(-NUM_EP // TEST_EVERY))
    best_score, best_run, temp_actor = -100000.0, 0, None
    r64 = torch.empty(1, dtype=torch.float64, device="cuda")
    for i in range(1, NUM_EP + 1):
        host_reset(env_train, ref_train, T, train_series.shape[1])
        reward_eps = np.float32(0); noise_eps = np.float32(0); ret_ref = 0.0
        for step in range(1, T + 1):
            noise = rng.normal(0, 0.1, (2, 1)).astype(np.float32)          # sample_noise(gn, rng_step + 1)
            s = env_train.state_tensor().clone()
            a, scaled = le.act(s, noise=dev(noise))
            r, s2 = env_train.step(scaled, reward64_out=r64)
            reward_eps = reward_eps + float(r64[0])                          # 0f0 + Float64 -> Float64 (DDPG.jl:190, :223)
            noise_eps = noise_eps + noise.mean(dtype=np.float32)
            memory.push(s, a, r, s2)                                         # remember(s, a, r, s′, finished)
            oa, osc = orc.act(ref_train.obs.copy(), noise=noise)
            s_ref = ref_train.obs.copy()
            r_ref, s2_ref, _ = ref_train.step(osc)
            ret_ref += float(r_ref[0])
            S = np.concatenate([S, s_ref], 1)[:, -MEM:]; A = np.concatenate([A, oa], 1)[:, -MEM:]
            R = np.concatenate([R, r_ref.astype(np.float32)])[-MEM:]; S2 = np.concatenate([S2, s2_ref], 1)[:, -MEM:]
            idx = rng.integers(0, len(memory), B).astype(np.int32)           # sample(MersenneTwister(rng_step), memory, BATCH_SIZE)
            le.replay(memory, n_updates=1, idx=idx)                          # replay(rng_rpl = rng_step)
            orc.update_batch(S[:, idx], A[:, idx], R[idx], S2[:, idx], np.zeros(B, np.float32))
            assert np.abs(a.cpu().numpy() - oa).max() < 2e-5, (i, step)
        total_reward[i - 1], noise_mean[i - 1] = reward_eps, noise_eps
        assert abs(float(reward_eps) - ret_ref) < 1e-3 * (abs(ret_ref) + 1)
        if i % TEST_EVERY == 1:
            k = -(-i // TEST_EVERY)
            score_all = 0.0
            for test_ep in range(1, TEST_RUNS + 1):
                host_reset(env_eval, ref_eval, 1439, eval_series.shape[1])   # maxsteps = 1439 of 1440 rows: always row 1, random Soc_b
                assert env_eval.idx[0] == 1
                score_all += float(le.rollout(env_eval, T)["ep_return"][0])
            score_mean[k - 1] = score_all / TEST_RUNS
            if score_mean[k - 1] > best_score:                                # saveBSON(actor, ...; idx = i, path = "temp")
                temp_actor = [le.get_layer(0, kk) for kk in range(3)]
                best_score, best_run = score_mean[k - 1], i
    assert best_run in (1, 3) and temp_actor is not None and np.isfinite(total_reward).all() and np.abs(noise_mean).max() > 0
    # the circular memory wrapped: the device ring and the host mirror still agree
    for got, want in zip(memory.get()[:4], (S, A, R, S2)):
        assert got.shape == want.shape
    np.testing.assert_allclose(memory.get()[0], S, rtol=1e-5, atol=1e-5)   # closed loop under actions that agree to ~1e-6
    # --- saveBSON(actor, ...) (driver :45) and, in the evaluating process, global actor = loadBSON(...) |> gpu; inference(track = 1)
    saved = [le.get_layer(0, k) for k in range(3)]
    fresh = sb.Learner()
    fresh.init(999)
    fresh.set_norm(s_min, s_max)
    for k in range(3):
        fresh.set_layer(0, k, *saved[k])
    env_eval.reset(rng=-1)
    out = fresh.rollout(env_eval, 1439, want_trace=True)
    assert out["trace"].shape == (1439, 23, 1) and float(out["trace"][-1, 0, 0]) == 1440.0
    ref_eval.reset(mode=0)
    score_ref = 0.0
    for t in range(1439):
        oa, osc = orc.act(ref_eval.obs.copy())
        r_ref, _, _ = ref_eval.step(osc)
        score_ref += float(r_ref[0])
    assert float(out["ep_return"][0]) == pytest.approx(score_ref, rel=1e-3)
    summary = sb.tracker.write_results_csv(str(tmp_path / "results.csv"), out["trace"])     # write_to_results_file
    assert summary["rewards"] == pytest.approx(float(out["ep_return"][0]), rel=1e-12)
    # --- inference(track < 0): the rule-based benchmark on the same data (driver :105)
    env_eval.reset(rng=-1)
    rb = env_eval.rollout(sb.POLICY_RULE, 1439, want_trace=True)
    assert rb["trace"].shape == (1439, 23, 1) and torch.isfinite(rb["ep_return"]).all()
