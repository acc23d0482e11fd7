"""Times prioritized replay (Learner.set_prioritized) against uniform replay, PER on and off alternated in one process, CUDA events:
  * update B = 120 (250/500, fp32): PER takes the tiled-GEMM sequence; beside it the tiled and the cluster-fused uniform updates;
  * update B = 8192 with the TF32 forward-chain kernels;
  * 80 learners at B = 120 (tensor cores on, BASELINE configs[4]);
  * the push-time refresh of the sum tree: one ddpg_episode step (64 instances, no update) and a 2^20-transition push into a
    24,000-record memory (replay_push: only the newest 24,000 survive, so every leaf is refreshed).
Each figure is the median over --reps alternations of --updates back-to-back updates (or pushes).  The card's name, power limit and
max SM clock are read in the same run.
usage: python tools/time_per.py [--reps 7] [--updates 200]   -> JSON lines"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import shems_b200 as sb  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=7)
ap.add_argument("--updates", type=int, default=200)
args = ap.parse_args()
assert torch.cuda.is_available(), "this measurement needs a CUDA device"
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                      text=True).stdout.strip()
rng = np.random.default_rng(0)


def filled(cap, n):
    m = sb.Replay(cap)
    s, s2 = torch.rand((9, n), device="cuda"), torch.rand((9, n), device="cuda")
    m.push(s, torch.rand((2, n), device="cuda") * 2 - 1, torch.rand(n, device="cuda") - 1, s2)
    m.enable_priorities()
    return m


def timed(fn, n):
    fn()   # warm-up (graph capture, module load)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / n


def update_case(name, P, B, tc, mem_cap=24_000, modes=("per", "tiled")):
    le = sb.Learner(params=sb.default_ddpg_params(population=P, batch=B, use_tensor_cores=tc))
    le.init(1)
    mems = [filled(mem_cap, mem_cap) for _ in range(P)]
    arg = mems[0] if P == 1 else mems
    U = args.updates if B < 1024 else max(args.updates // 4, 20)

    def run(mode):
        if mode == "per":
            le.set_prioritized(0.6, 0.4, 1e-6)
        else:
            le.set_prioritized(None)
            le.set_fused(mode == "fused")
        return timed(lambda: le.replay(arg, rng_rpl=3, n_updates=U), U)

    res = {m: [] for m in modes}
    for _ in range(args.reps):
        for m in modes:
            res[m].append(run(m))
    out = dict(case=name, card=card, learners=P, batch=B, tc=tc, updates_per_sample=U, reps=args.reps)
    for m in modes:
        out[f"{m}_us"] = float(np.median(res[m]))
        out[f"{m}_range_us"] = [float(np.min(res[m])), float(np.max(res[m]))]
    out["per_overhead_vs_tiled"] = out["per_us"] / out["tiled_us"] - 1.0
    print(json.dumps(out), flush=True)


update_case("update_B120", 1, 120, 0, modes=("per", "tiled", "fused"))
update_case("update_B8192_chain", 1, 8192, 1)
update_case("population_80x120", 80, 120, 1, mem_cap=24_000)

# push-time refresh: one ddpg_episode step of 64 instances into a 24,000-record memory, no update
ser = sb.series.synth_charger98(4320, seed=98)
env = sb.Shems(72, ser, n_envs=64)
le = sb.Learner()
le.init(1)
steps = 72
res = {"per": [], "plain": []}
for _ in range(args.reps):
    for mode in res:
        mem = filled(24_000, 24_000) if mode == "per" else sb.Replay(24_000)
        if mode == "per":
            le.set_prioritized(0.6, 0.4, 1e-6)
        else:
            le.set_prioritized(None)
            mem.push(torch.rand((9, 24_000), device="cuda"), torch.rand((2, 24_000), device="cuda"), torch.rand(24_000, device="cuda"),
                     torch.rand((9, 24_000), device="cuda"))

        def ep():
            env.reset(rng=1)
            le.episode(env, mem, steps, train=True, rng_ep=1, updates_per_step=0)
        res[mode].append(timed(ep, steps))
print(json.dumps(dict(case="episode_step_64_no_update", card=card, per_us=float(np.median(res["per"])), plain_us=float(np.median(res["plain"])),
                      refresh_us=float(np.median(res["per"]) - np.median(res["plain"])))), flush=True)

n = 1 << 20
big = [torch.rand((9, n), device="cuda"), torch.rand((2, n), device="cuda"), torch.rand(n, device="cuda"), torch.rand((9, n), device="cuda")]
res = {"per": [], "plain": []}
mems = {"per": filled(24_000, 24_000), "plain": sb.Replay(24_000)}
for _ in range(args.reps):
    for mode, mem in mems.items():
        res[mode].append(timed(lambda: [mem.push(*big) for _ in range(10)], 10))
print(json.dumps(dict(case="push_2^20_into_24000", card=card, per_us=float(np.median(res["per"])), plain_us=float(np.median(res["plain"])),
                      refresh_us=float(np.median(res["per"]) - np.median(res["plain"])))), flush=True)
