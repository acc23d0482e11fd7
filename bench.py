#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W          (N > 1: launched under torch.distributed.run)
    python bench.py --impl reference ...                    (the CPU arm: the oracle port on all host cores)
    python bench.py ... --dump-outputs DIR                  (also writes the last timed step's outputs as DIR/<name>.npy)

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): shems_LU1 random-action
rollout, 2^20 instances per GPU x 8760 hourly steps on a synthetic ChargerID98-shaped 8761-row year series,
every transition (s, a, r, s', done) written into the device-resident replay ring as populate_memory does
(memory_plotting_saving.jl:9-29).  One bench "step" = one reset + one fused 8760-step rollout of all instances.
Instances shard across ranks with no collective (global env id keys the RNG), per-GPU work fixed: "weak".  For N > 1 the line
also carries `strong_scaling`: configs[2] as written, 2^20 instances in TOTAL split over the ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "shems_LU1 env-steps/s (batched)"
UNIT = "env-steps/s"
DTYPE = "f32/f64 mixed (Julia promotion rules)"
WORKLOAD = "BASELINE configs[2]: shems_LU1 random-action rollout writing replay transitions"
ALG_BYTES_PER_ENV_STEP = 88  # s 36 + a 8 + r 4 + s' 36 + done 4 (SURVEY.md §8d, rollout writing replay transitions)


# stdout carries exactly ONE line, the JSON: everything libraries print there (NCCL's version banner under NCCL_DEBUG, ...) is sent
# to stderr by pointing file descriptor 1 at stderr for the whole run; emit() writes the line to the real stdout
_REAL_STDOUT = None


def _quiet_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=1 << 20)
    ap.add_argument("--horizon", type=int, default=8760)
    ap.add_argument("--ring-slots", type=int, default=16, help="replay ring capacity in multiples of envs-per-gpu")
    ap.add_argument("--cpu-sample-envs", type=int, default=0, help="0: auto-size the CPU sample to ~15 s")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-ddpg", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    return args


# ------------------------------------------------------------------------------ CPU arm (oracle port)
def cpu_rollout_rate(ser, horizon, n_envs, seed=1):
    """env-steps/s of the CPU oracle (OpenMP over instances, all host cores) on n_envs x horizon steps."""
    from oracle import oracle as O
    O.set_threads(cpu_cores())
    P = O.params_for_charger(98)
    env = O.OracleEnv(P, ser, horizon, n_envs)
    env.reset(mode=2, seed=seed)
    t0 = time.perf_counter()
    env.rollout(1, horizon, seed=seed)
    dt = time.perf_counter() - t0
    return n_envs * horizon / dt, dt


def cpu_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_baseline(ser, horizon, sample_envs=0, target_s=15.0):
    cores = cpu_cores()
    os.environ.setdefault("OMP_NUM_THREADS", str(cores))
    if sample_envs <= 0:
        probe = max(cores * 2, 16)
        rate, dt = cpu_rollout_rate(ser, horizon, probe)
        sample_envs = int(max(probe, min(1 << 20, target_s * rate / horizon)))
        sample_envs = (sample_envs // cores) * cores or cores
    rate, dt = cpu_rollout_rate(ser, horizon, sample_envs)
    return dict(value=rate, unit=UNIT, cores=cores, kind="port",
                sample=f"{sample_envs} instances x {horizon} steps (same series, same Philox actions), OpenMP over instances, {dt:.1f} s; "
                       "the reference's Julia cannot run here (not installed), this is the repo's C restatement of it; it accumulates the episode returns but "
                       "does not write the 88-byte transitions, i.e. it does LESS work per step than the GPU arm"), dt


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path = the oracle port (Julia is not installed)."""
    if rank != 0:
        return
    import shems_b200 as sb
    ser = sb.series.synth_charger98(args.horizon + 1, seed=98)
    cores = cpu_cores()
    os.environ.setdefault("OMP_NUM_THREADS", str(cores))
    probe_rate, _ = cpu_rollout_rate(ser, args.horizon, max(cores * 2, 16))
    per_step_s = min(20.0, 120.0 / max(1, args.steps + args.warmup))
    n = int(max(cores, per_step_s * probe_rate / args.horizon))
    n = (n // cores) * cores or cores
    for _ in range(args.warmup):
        cpu_rollout_rate(ser, args.horizon, n)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_rollout_rate(ser, args.horizon, n)
    dt = time.perf_counter() - t0
    value = args.steps * n * args.horizon / dt
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * dt / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype=DTYPE,
                data="synthetic", impl="reference",
                # the b200 arm's workload; the CPU arm runs a bounded sample of its instances per step (cpu_baseline.sample)
                config=dict(workload=WORKLOAD, envs_per_gpu=args.envs_per_gpu, envs_total=args.envs_per_gpu * world, horizon=args.horizon,
                            series_rows=args.horizon + 1, charger=98, sample_envs_per_step=n,
                            note="the same rollout (same series, same Philox action streams) on the host cores, a bounded sample of the instances per step"),
                cpu_baseline=dict(value=value, unit=UNIT, cores=cores, kind="port",
                                  sample=f"{n} instances x {args.horizon} steps per step, OpenMP over instances; returns only (no transition writes: less work than the GPU arm)"),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    emit(line)


# ------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self._halt = threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------ GPU arm
def ddpg_updates_per_s(sb, torch, ser_train, n_updates=2000):
    """DDPG updates/s at the reference's tuned config (B=120, MEM=24,000, 250/500) — reported beside the env metric."""
    env = sb.Shems(72, ser_train, n_envs=1000)
    mem = sb.Replay(24_000)
    for ep in range(1):
        env.reset(rng=ep + 1)
        env.rollout(sb.POLICY_RANDOM, 24, seed=ep + 1, replay=mem, want_return=False)
    mn, mx = mem.min_max_buffer(24_000, rng_mm=1)

    def timed(fused):
        le = sb.Learner()
        le.set_fused(fused)
        le.init(1)
        le.set_norm(mn, mx)
        le.replay(mem, rng_rpl=1, n_updates=50)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        le.replay(mem, rng_rpl=2, n_updates=n_updates)
        e1.record()
        torch.cuda.synchronize()
        le.close()
        return e0.elapsed_time(e1)

    ms = timed(True)          # the default: two thread-block-cluster kernels per update (csrc/ddpg_fused.cu)
    ms_tiled = timed(False)   # one launch per matrix product (the path populations and large batches use)
    return dict(updates_per_s=n_updates / (ms * 1e-3), us_per_update=1e3 * ms / n_updates, batch=120, l1=250, l2=500, mem=24_000,
                kernels_per_update=4, flops_per_update=3.078e8, path="cluster-fused (critic pass incl. minibatch gather, ADAM, actor pass, ADAM+Polyak)",
                tiled_gemm_path=dict(updates_per_s=n_updates / (ms_tiled * 1e-3), us_per_update=1e3 * ms_tiled / n_updates, kernels_per_update=21))


def ddpg_cpu_baseline(torch, batch=120, l1=250, l2=500, n_updates=200, gamma=0.99, tau=1e-3):
    """replay() (DDPG.jl:121-145) restated with torch on the host cores — what the reference's Flux/Zygote update costs on a CPU
    (Julia is not installed; a baseline, not the target).  Same nets, losses, ADAM(1e-4 / 1e-3), Polyak."""
    import torch.nn as nn
    cores = cpu_cores()
    torch.set_num_threads(cores)

    def mlp(i, o, last):
        return nn.Sequential(nn.Linear(i, l1), nn.ReLU(), nn.Linear(l1, l2), nn.ReLU(), nn.Linear(l2, o), last)

    actor, critic = mlp(9, 2, nn.Tanh()), mlp(11, 1, nn.Identity())
    actor_t, critic_t = mlp(9, 2, nn.Tanh()), mlp(11, 1, nn.Identity())
    actor_t.load_state_dict(actor.state_dict()); critic_t.load_state_dict(critic.state_dict())
    oa, oc = torch.optim.Adam(actor.parameters(), lr=1e-4, eps=1e-8), torch.optim.Adam(critic.parameters(), lr=1e-3, eps=1e-8)
    g = torch.Generator().manual_seed(0)
    mem = [torch.rand((24_000, k), generator=g) for k in (9, 2, 1, 9)]

    def update():
        idx = torch.randint(0, 24_000, (batch,), generator=g)
        s, a, r, s2 = (m[idx] for m in mem)
        with torch.no_grad():
            y = r + gamma * critic_t(torch.cat([s2, actor_t(s2)], 1))
        lc = ((critic(torch.cat([s, a], 1)) - y) ** 2).mean()
        oc.zero_grad(); lc.backward(); oc.step()
        la = -critic(torch.cat([s, actor(s)], 1)).mean()
        oa.zero_grad(); la.backward(); oa.step()
        with torch.no_grad():
            for t, m in ((actor_t, actor), (critic_t, critic)):
                for pt, pm in zip(t.parameters(), m.parameters()):
                    pt.mul_(1 - tau).add_(pm, alpha=tau)

    t0 = time.perf_counter()
    for _ in range(5):
        update()
    per = (time.perf_counter() - t0) / 5
    n_updates = int(max(5, min(n_updates, 4.0 / max(per, 1e-6))))     # bounded: about 4 s of CPU work
    t0 = time.perf_counter()
    for _ in range(n_updates):
        update()
    dt = time.perf_counter() - t0
    return dict(updates_per_s=n_updates / dt, us_per_update=1e6 * dt / n_updates, threads=cores, kind="port",
                what="torch-CPU restatement of replay() at B=%d, %d/%d" % (batch, l1, l2))


def ddpg_large_batch(sb, torch, ser_train, batch=8192, n_updates=100):
    """DDPG updates/s where batch x width is a dense contraction (BASELINE configs[3], 8192 parallel instances): the 250x500
    products run on the TF32 tcgen05 kernel; tensor-pipe evidence in profiles/."""
    env = sb.Shems(72, ser_train, n_envs=8192)
    mem = sb.Replay(1 << 20)
    env.reset(rng=1)
    env.rollout(sb.POLICY_RANDOM, 72, seed=1, replay=mem, want_return=False)
    out = {}
    for name, tc in (("tf32_tcgen05", 1), ("fp32_simt", 0)):
        le = sb.Learner(params=sb.default_ddpg_params(batch=batch, use_tensor_cores=tc))
        le.init(1)
        mn, mx = mem.min_max_buffer(24_000, rng_mm=1)
        le.set_norm(mn, mx)
        le.replay(mem, rng_rpl=1, n_updates=10)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        le.replay(mem, rng_rpl=2, n_updates=n_updates)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        out[name] = dict(updates_per_s=n_updates / (ms * 1e-3), us_per_update=1e3 * ms / n_updates, samples_per_s=batch * n_updates / (ms * 1e-3),
                         tflops=10 * 256_500 * batch * n_updates / (ms * 1e-3) / 1e12)
        le.close()
    out.update(batch=batch, l1=250, l2=500, flops_per_update=10 * 256_500 * batch)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    bf16 = float(json.load(open(peaks_path))["bf16_tflops"]) if os.path.exists(peaks_path) else 1665.0
    # TF32 dense tensor rate = half the bf16 rate; the update's algorithmic FLOPs (SURVEY §8d) over its whole duration, thin
    # streaming kernels and ADAM included — see DESIGN §4.4(ii) for why K = 250 products sit far below the tensor peak
    out["roofline"] = dict(bound="tensor", achieved=out["tf32_tcgen05"]["tflops"], peak=bf16 / 2, unit="TFLOP/s",
                           frac=out["tf32_tcgen05"]["tflops"] / (bf16 / 2), peak_source="MEASURED_PEAKS.json bf16_tflops / 2 (TF32 dense)",
                           note="whole replay() incl. streaming kernels and ADAM; the 250x500 products alone: profiles/r1_tc_gemm.md")
    return out


def rule_based_config2(sb, torch, ser_train, n_envs=4096, T=72, reps=50):
    """BASELINE configs[1]: the rule-based controller (`track = -0.5`) on 4096 instances x 72 steps, one fused launch per episode:
    0.26 MB per step — latency-bound by construction (SURVEY §8d), reported as a time."""
    env = sb.Shems(T, ser_train, n_envs=n_envs)
    for _ in range(3):
        env.reset(rng=-1)
        env.rollout(sb.POLICY_RULE, T)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        env.reset(rng=-1)
        out = env.rollout(sb.POLICY_RULE, T)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    return dict(envs=n_envs, steps=T, us_per_episode_batch=1e3 * ms, env_steps_per_s=n_envs * T / (ms * 1e-3),
                mean_return=float(out["ep_return"].mean()), note="reset!(rng=-1) + one fused 72-step launch; launch/latency bound")


def reference_training_loop(sb, torch, ser_train, episodes=30):
    """BASELINE configs[0], the reference's own training loop (DDPG_reinforce_charger_v1.jl: ONE instance, EP_LENGTH = 72, BATCH = 120,
    MEM = 24,000, 250/500): episode! = act -> step! -> remember -> replay() per step, through the native `ddpg_episode` loop."""
    env = sb.Shems(72, ser_train, n_envs=1)
    le = sb.Learner()
    le.init(1231)
    drv = sb.Driver(env, None, learner=le, mem_size=24_000, ep_length=72, sigma=0.1, updates_per_step=1, rng_run=1231)
    drv.populate_memory()
    drv.min_max_buffer()
    for ep in range(3):
        drv.episode(env, train=True, rng_ep=ep + 1)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for ep in range(episodes):
        drv.episode(env, train=True, rng_ep=100 + ep)
    e1.record()
    torch.cuda.synchronize()
    steps = episodes * 72
    ms = e0.elapsed_time(e1)
    return dict(instances=1, batch=120, mem=24_000, episodes_timed=episodes, training_steps_per_s=steps / (ms * 1e-3), us_per_step=1e3 * ms / steps,
                full_run_seconds=72_072 * ms / steps * 1e-3,
                note="one step = cluster-fused act kernel, step!, remember/return kernel, 4-kernel replay(); full_run = 1001 episodes x 72 steps")


def rollout_returns_only(sb, torch, ser, n_envs=1 << 20, T=2000, reps=3):
    """The same random-action rollout with the episode returns as its only output (8 B per instance per launch): no HBM roofline
    applies (SURVEY §8d) — this is the arithmetic ceiling of the Julia-exact step, reported as env-steps/s."""
    env = sb.Shems(T, ser, n_envs=n_envs)
    env.reset(rng=1)
    env.rollout(sb.POLICY_RANDOM, T, seed=1)
    torch.cuda.synchronize()
    ms = []
    for rep in range(reps):
        env.reset(rng=2 + rep)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        env.rollout(sb.POLICY_RANDOM, T, seed=2 + rep)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    t = sorted(ms)[len(ms) // 2]
    return dict(envs=n_envs, steps=T, env_steps_per_s=n_envs * T / (t * 1e-3), ms_per_launch=t,
                note="no per-step sink: bound by instruction issue, not by bytes")


POP_CHARGERS = (1, 2, 3, 4, 5, 6, 7, 8, 9, 98)  # capacities of shems_LU1.jl:47-59; 10 chargers x 64 seeds = 640 learners on 8 GPUs


def ddpg_population(sb, torch, dist, rank, world, ser_train, per_gpu=80, n_updates=40, tc=1, n_envs=64, episodes=3):
    """BASELINE configs[4]: independent-seed learners (the reference's one-process-per-seed parallelism), per_gpu of them per
    rank advanced by the same launches; learner g = rank*per_gpu + l trains charger POP_CHARGERS[(g // 64) % 10] with seed g.
    Two numbers: replay() alone (learner_updates_per_s) and the whole training loop act -> step! -> remember -> replay()
    (train_learner_updates_per_s; every learner steps n_envs instances of its own charger, all in one environment handle).
    No collective during training (SURVEY §8e); rank 0 gathers the rates."""
    dev = torch.cuda.current_device()
    from shems_b200 import sharding
    if per_gpu * world == 640:          # the full configs[4] population: 10 chargers x 64 seeds
        gids, chargers, seeds = sharding.population_shard(rank, world)
    else:                               # fewer GPUs: the first per_gpu*world learners of it
        gids = [rank * per_gpu + l for l in range(per_gpu)]
        chargers = [POP_CHARGERS[(g // 64) % len(POP_CHARGERS)] for g in gids]
        seeds = [int("123%d" % (g % 64 + 1)) for g in gids]
    drv = sb.PopulationDriver(ser_train, chargers=chargers, seeds=[1000 * g + s for g, s in zip(gids, seeds)], n_envs=n_envs, device=dev,
                              use_tensor_cores=tc)
    drv.populate_memory()
    drv.min_max_buffer()
    le, mems = drv.learner, drv.mems
    le.replay(mems, rng_rpl=7, n_updates=5)

    def timed(fn):
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ms = timed(lambda: le.replay(mems, rng_rpl=11, n_updates=n_updates))
    drv.episode(train=True, rng_ep=1)
    ms_train = timed(lambda: [drv.episode(train=True, rng_ep=2 + e) for e in range(episodes)])
    lc, la = le.select(0).losses()
    steps = episodes * drv.ep_length
    return dict(learners=per_gpu * world, learners_per_gpu=per_gpu, chargers=sorted({POP_CHARGERS[(g // 64) % 10] for g in range(per_gpu * world)}),
                batch=120, l1=250, l2=500, precision="tf32 products, fp32 accumulate" if tc else "fp32",
                learner_updates_per_s=per_gpu * world * n_updates / (ms * 1e-3), us_per_population_update=1e3 * ms / n_updates,
                tflops=10 * 256_500 * 120 * per_gpu * world * n_updates / (ms * 1e-3) / 1e12,
                train_learner_updates_per_s=per_gpu * world * steps / (ms_train * 1e-3), train_us_per_vector_step=1e3 * ms_train / steps,
                train_env_steps_per_s=per_gpu * world * n_envs * steps / (ms_train * 1e-3), envs_per_learner=n_envs,
                collective="none (independent seeds)", loss_crit_learner0=lc, loss_act_learner0=la)


def ddpg_dp_updates_per_s(sb, torch, dist, rank, ser_train, n_updates=300):
    """Data-parallel learner: every rank samples its own replay shard (B=120 each); the critic and actor gradients are averaged
    over the ranks twice per update.  Two implementations are timed: `nccl` (ddpg_update_phase + two NCCL all-reduces issued
    from the host) and `fused_peer` (ddpg_update_dp: the exchange runs inside the ADAM kernels over NVLink peer memory, the
    whole update is one captured graph)."""
    dev = torch.cuda.current_device()
    env = sb.Shems(72, ser_train, n_envs=1000, device=dev, env_id_base=rank * 1000)
    mem = sb.Replay(24_000, device=dev)
    env.reset(rng=1)
    env.rollout(sb.POLICY_RANDOM, 24, seed=1, replay=mem, want_return=False)
    mn, mx = mem.min_max_buffer(24_000, rng_mm=1)
    out = dict(global_batch=120 * dist.get_world_size())

    def in_sync(le):
        w0 = torch.from_numpy(le.get_layer(0, 1)[0]).cuda()
        ref = w0.clone()
        dist.broadcast(ref, 0)
        ok = torch.tensor([float(torch.equal(w0, ref))], device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        return bool(ok.item() == 1.0)

    def timed(fn):
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    le = sb.Learner(device=dev)
    le.init(1)                                   # identical replicas on every rank
    le.set_norm(mn, mx)
    for u in range(20):
        le.replay_dp(mem, rng_rpl=100 + rank, dist=dist)
    ms = timed(lambda: [le.replay_dp(mem, rng_rpl=1000 + rank, dist=dist) for _ in range(n_updates)])
    out["nccl"] = dict(updates_per_s=n_updates / (ms * 1e-3), us_per_update=1e3 * ms / n_updates,
                       allreduce_bytes_per_update=4 * int(le.grad_tensor().numel()), replicas_bit_identical=in_sync(le))
    le.close()
    try:
        lf = sb.Learner(device=dev)
        lf.init(1)
        lf.set_norm(mn, mx)
        lf.dp_connect_dist(dist)
        dist.barrier()
        lf.replay_fused_dp(mem, rng_rpl=100 + rank, n_updates=20)
        ms = timed(lambda: lf.replay_fused_dp(mem, rng_rpl=1000 + rank, n_updates=n_updates))
        out["fused_peer"] = dict(updates_per_s=n_updates / (ms * 1e-3), us_per_update=1e3 * ms / n_updates, exchange_status=lf.dp_status(),
                                 peer_bytes_pushed_per_update=4 * int(lf.grad_tensor().numel()) * (dist.get_world_size() - 1),
                                 replicas_bit_identical=in_sync(lf))
    except Exception as e:
        out["fused_peer"] = dict(error=str(e))
    return out


DUMP_SAMPLE = 1 << 18   # instances and replay rows --dump-outputs writes at most: ~41 MB in all


def dump_outputs(dirname, env, mem, out):
    """--dump-outputs: what the last timed step left its caller, as float32 / float64 DIR/<name>.npy — episode return, state and row
    index of a fixed seeded sample of the instances, and the transitions at a fixed seeded sample of the replay ring's logical
    indices (0 = oldest).  The same arguments give the same inputs, so two builds can be compared array by array."""
    os.makedirs(dirname, exist_ok=True)
    rng = np.random.default_rng(0)
    envs = np.sort(rng.choice(env.n_envs, min(env.n_envs, DUMP_SAMPLE), replace=False))
    rows = np.sort(rng.choice(len(mem), min(len(mem), DUMP_SAMPLE), replace=False)).astype(np.int32)
    s, a, r, s2, done = (x.cpu().numpy() for x in mem.sample(len(rows), idx=rows))
    arrays = dict(env_ids=envs.astype(np.float64), ep_return=out["ep_return"].cpu().numpy()[envs], state=env.state[:, envs],
                  state_idx=env.idx[envs].astype(np.float64), replay_rows=rows.astype(np.float64), replay_s=s, replay_a=a, replay_r=r,
                  replay_s2=s2, replay_done=done)
    for name, x in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), x)


def main():
    args = parse()
    _quiet_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import shems_b200 as sb

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n, T = args.envs_per_gpu, args.horizon
    ser = sb.series.synth_charger98(T + 1, seed=98)
    from shems_b200 import sharding
    env_base, _ = sharding.weak_range(n, rank)
    env = sb.Shems(T, ser, n_envs=n, device=local_rank, env_id_base=env_base)
    mem = sb.Replay(n * args.ring_slots, device=local_rank)
    # e2e inputs: the two reset draws per instance come from pinned HOST memory every step (H2D inside the timed region),
    # the per-instance episode return is read back to pinned HOST memory every step (D2H inside the timed region)
    rng = np.random.default_rng(1234 + rank)
    idx0_pin = torch.ones(n, dtype=torch.int32).pin_memory()          # nrows - maxsteps == 1: the only admissible start row
    socb0_pin = torch.from_numpy(rng.uniform(0, 6.75, n).astype(np.float32)).pin_memory()
    ret_pin = torch.empty(n, dtype=torch.float64).pin_memory()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    kernel_ms = []

    def device_step(seed, timed):
        env.reset(rng=seed)                      # reset kernel (Philox draws on the device)
        if timed:
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0.record()
        out = env.rollout(sb.POLICY_RANDOM, T, seed=seed, replay=mem, want_return=True)
        if timed:
            k1.record()
            kernel_ms.append((k0, k1))
        return out

    def e2e_step(seed):
        env.reset(idx0=idx0_pin.numpy(), socb0=socb0_pin.numpy())     # H2D of the host draws + reset kernel
        out = env.rollout(sb.POLICY_RANDOM, T, seed=seed, replay=mem, want_return=True)
        ret_pin.copy_(out["ep_return"], non_blocking=True)            # D2H of the step's result
        torch.cuda.current_stream().synchronize()
        return float(ret_pin[0])

    # ---- device-resident throughput (`value`) ----
    for w in range(args.warmup):
        device_step(100 + w, False)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = int(sb._lib.lib().shems_env_kernel_launches())
    ev[0].record()
    for k in range(args.steps):
        out = device_step(1000 + k, True)
    ev[1].record()
    launches_timed = int(sb._lib.lib().shems_env_kernel_launches()) - launches0   # counted by the library at its launch sites
    barrier()
    ms = ev[0].elapsed_time(ev[1])
    if args.dump_outputs and rank == 0:        # before the e2e steps below overwrite the environment and the ring
        dump_outputs(args.dump_outputs, env, mem, out)
    # ---- end-to-end through the public API with host buffers (`e2e`) ----
    for w in range(max(1, args.warmup // 2)):
        e2e_step(200 + w)
    barrier()
    ev[2].record()
    for k in range(args.steps):
        e2e_step(2000 + k)
    ev[3].record()
    barrier()
    ms_e2e = ev[2].elapsed_time(ev[3])
    clocks = sampler.stop()
    kern = [a.elapsed_time(b) for a, b in kernel_ms]
    t = torch.tensor([ms, ms_e2e, float(np.mean(kern))], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e, kern_ms = (float(x) for x in t.cpu())
    total_steps = float(world) * n * T * args.steps
    value = total_steps / (ms * 1e-3)
    e2e_value = total_steps / (ms_e2e * 1e-3)

    # ---- BASELINE configs[2] as written: 2^20 instances in TOTAL, sharded over the ranks (strong scaling; N > 1 only) ----
    strong = None
    if world > 1:
        total = args.envs_per_gpu
        lo, cnt = sharding.shard_range(total, rank, world)
        env_s = sb.Shems(T, ser, n_envs=cnt, device=local_rank, env_id_base=lo)

        def strong_step(seed):
            env_s.reset(rng=seed)
            env_s.rollout(sb.POLICY_RANDOM, T, seed=seed, replay=mem, want_return=True)
        for w in range(args.warmup):
            strong_step(300 + w)
        barrier()
        es = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        es[0].record()
        for k in range(args.steps):
            strong_step(3000 + k)
        es[1].record()
        barrier()
        ts = torch.tensor([es[0].elapsed_time(es[1])], dtype=torch.float64, device="cuda")
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        ms_s = float(ts.item())
        strong = dict(scaling="strong", envs_total=total, envs_per_gpu=cnt, value=float(total) * T * args.steps / (ms_s * 1e-3), unit=UNIT,
                      ms_per_step=ms_s / args.steps, vs_weak_value=float(total) * T * args.steps / (ms_s * 1e-3) / value,
                      note="2^20 instances in total (configs[2] as written), contiguous env-id ranges per rank, no collective; vs_weak_value = "
                           "this throughput / the weak-scaling value of the same run (1.0 = no loss from the smaller per-GPU grids)")
        env_s.close()

    ddpg_dp = ddpg_pop = None
    if not args.skip_ddpg:
        mem.close()                       # the 1.5 GB ring is no longer needed
        env.close()
        ser_train = sb.series.synth_charger98(4320, seed=98)
        if dist is not None:
            try:
                ddpg_dp = ddpg_dp_updates_per_s(sb, torch, dist, rank, ser_train)
            except Exception as e:
                ddpg_dp = dict(error=str(e))
        try:
            ddpg_pop = ddpg_population(sb, torch, dist, rank, world, ser_train)
        except Exception as e:
            ddpg_pop = dict(error=str(e))
    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    achieved = ALG_BYTES_PER_ENV_STEP * n * T / (kern_ms * 1e-3) / 1e9
    # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed `ncu --set full` capture, scaled per env-step
    traffic = traffic_src = None
    tpath = os.path.join(ROOT, "profiles", "r2_rollout_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic = tj["dram_bytes_per_env_step"] * n * T
        traffic_src = f"profiles/r2_rollout_traffic.json: {tj['dram_bytes_per_env_step']:.2f} DRAM B/env-step ({tj['capture']}) x env-steps of this launch"
    roofline = dict(bound="hbm", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak, traffic=traffic, traffic_source=traffic_src,
                    kernel="shems_rollout_kernel<POLICY_RANDOM, no trace, FAST>", kernel_ms=kern_ms,
                    algorithmic_bytes_per_launch=ALG_BYTES_PER_ENV_STEP * n * T, peak_source=peak_src)
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=ms / args.steps,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype=DTYPE, data="synthetic",
                config=dict(workload=WORKLOAD,
                            envs_per_gpu=n, envs_total=n * world, horizon=T, series_rows=T + 1, charger=98,
                            replay_ring_transitions=n * args.ring_slots, bytes_per_env_step=ALG_BYTES_PER_ENV_STEP,
                            l2_policy=f"working set per launch {ALG_BYTES_PER_ENV_STEP * n * args.ring_slots / 1e6:.0f} MB of ring >> 126 MB L2 (no flush needed)",
                            parallelism=f"env-sharded x{world}, no collective"),
                roofline=roofline, clocks=clocks,
                e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=int(8 * n), d2h_bytes_per_step=int(8 * n),
                         note="reset draws (idx0, Soc_b0) from pinned host memory and episode returns back to pinned host memory every step"),
                gpu_launches=launches_timed)
    if not args.skip_ddpg:
        try:
            line["ddpg"] = ddpg_updates_per_s(sb, torch, sb.series.synth_charger98(4320, seed=98))
        except Exception as e:  # never lose the env number to the secondary metric
            line["ddpg"] = dict(error=str(e))
        try:
            line["reference_training_loop"] = reference_training_loop(sb, torch, sb.series.synth_charger98(4320, seed=98))
        except Exception as e:
            line["reference_training_loop"] = dict(error=str(e))
        try:
            line["rollout_returns_only"] = rollout_returns_only(sb, torch, ser)
        except Exception as e:
            line["rollout_returns_only"] = dict(error=str(e))
        try:
            line["rule_based_4096x72"] = rule_based_config2(sb, torch, sb.series.synth_charger98(4320, seed=98))
        except Exception as e:
            line["rule_based_4096x72"] = dict(error=str(e))
        try:
            line["ddpg_large_batch"] = ddpg_large_batch(sb, torch, sb.series.synth_charger98(4320, seed=98))
        except Exception as e:
            line["ddpg_large_batch"] = dict(error=str(e))
    if strong is not None:
        line["strong_scaling"] = strong
    if ddpg_dp is not None:
        line["ddpg_data_parallel"] = ddpg_dp
    if ddpg_pop is not None:
        line["ddpg_population"] = ddpg_pop
    if not args.skip_cpu_baseline and world == 1:   # the CPU baselines are timed on rank 0 at N = 1 only
        cb, _ = cpu_baseline(ser, T, args.cpu_sample_envs)
        line["cpu_baseline"] = cb
        if not args.skip_ddpg and isinstance(line.get("ddpg"), dict):
            try:
                line["ddpg"]["cpu_baseline"] = ddpg_cpu_baseline(torch)
            except Exception as e:
                line["ddpg"]["cpu_baseline"] = dict(error=str(e))
    emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
