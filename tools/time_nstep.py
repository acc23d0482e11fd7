"""Times n-step returns (Learner.set_nstep) in one process, n = 1, 3, 8, 16 alternated, CUDA events:
  * update B = 120 (250/500, fp32), cluster-fused and tiled;
  * update B = 8192 with the TF32 forward-chain kernels;
  * 80 learners at B = 120 (tensor cores on, BASELINE configs[4]);
  * the successor-link pass, with and without links: one ddpg_episode step (64 instances, no update), one rollout step of 2^20
    instances into a 2^20-record memory (a rollout cannot write more instances than its memory holds), and a 2^20-transition push
    into a 24,000-record memory (only the newest 24,000 survive and are linked).
The update memories hold 24,000 records of random-policy rollouts (1,000 instances x 24 steps), so the rows walk real chains.  Each
figure is the median over --reps alternations of --updates back-to-back updates.  The card's name, power limit and max SM clock are
read in the same run.
usage: python tools/time_nstep.py [--reps 7] [--updates 200]   -> JSON lines"""
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
ser = sb.series.synth_charger98(4320, seed=98)
NS = (1, 3, 8, 16)


def fill(cap, seed, links=True):
    """a cap-record memory of random-policy rollouts: 1,000 instances, 24 steps each (every instance a chain of 24 records)"""
    m = sb.Replay(cap)
    if links:
        m.enable_successors()
    env = sb.Shems(24, ser, n_envs=cap // 24)
    env.reset(rng=seed)
    env.rollout(sb.POLICY_RANDOM, 24, seed=seed, replay=m, want_return=False)
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


def update_case(name, P, B, tc, fused=True):
    le = sb.Learner(params=sb.default_ddpg_params(population=P, batch=B, use_tensor_cores=tc))
    le.init(1)
    le.set_fused(fused)
    mems = [fill(24_000, 10 + l) for l in range(P)]
    arg = mems[0] if P == 1 else mems
    for l, m in enumerate(mems):
        le.select(l).set_norm(*m.min_max_buffer(len(m), rng_mm=1))
    le.select(0)
    U = args.updates if B < 1024 else max(args.updates // 4, 20)
    res = {n: [] for n in NS}
    for _ in range(args.reps):
        for n in NS:
            le.set_nstep(n)
            res[n].append(timed(lambda: le.replay(arg, rng_rpl=3, n_updates=U), U))
    out = dict(case=name, card=card, learners=P, batch=B, tc=tc, fused=le.set_fused(fused), updates_per_sample=U, reps=args.reps)
    for n in NS:
        out[f"n{n}_us"] = float(np.median(res[n]))
        out[f"n{n}_range_us"] = [float(np.min(res[n])), float(np.max(res[n]))]
    print(json.dumps(out), flush=True)


update_case("update_B120_fused", 1, 120, 0, fused=True)
update_case("update_B120_tiled", 1, 120, 0, fused=False)
update_case("update_B8192_chain", 1, 8192, 1)
update_case("population_80x120", 80, 120, 1)

# the link pass: one ddpg_episode step of 64 instances into a 24,000-record memory, no update
env = sb.Shems(72, ser, n_envs=64)
le = sb.Learner()
le.init(1)
steps = 72
res = {"links": [], "plain": []}
for _ in range(args.reps):
    for mode in res:
        mem = fill(24_000, 5, links=(mode == "links"))

        def ep():
            env.reset(rng=1)
            le.episode(env, mem, steps, train=True, rng_ep=1, updates_per_step=0)
        res[mode].append(timed(ep, steps))
print(json.dumps(dict(case="episode_step_64_no_update", card=card, links_us=float(np.median(res["links"])), plain_us=float(np.median(res["plain"])),
                      link_pass_us=float(np.median(res["links"]) - np.median(res["plain"])))), flush=True)

# one rollout step of 2^20 instances into a 2^20-record memory: the pass links every record to the one 2^20 before it (none survive)
big = sb.Shems(1, ser, n_envs=1 << 20)
res = {"links": [], "plain": []}
mems = {"links": sb.Replay(1 << 20).enable_successors(), "plain": sb.Replay(1 << 20)}
small = {"links": sb.Replay(24_000).enable_successors(), "plain": sb.Replay(24_000)}
for _ in range(args.reps):
    for mode in res:
        def roll():
            for _ in range(10):
                big.reset(rng=2)
                big.rollout(sb.POLICY_RANDOM, 1, seed=2, replay=mems[mode], want_return=False)
        res[mode].append(timed(roll, 10))
print(json.dumps(dict(case="rollout_step_2^20", card=card, links_us=float(np.median(res["links"])), plain_us=float(np.median(res["plain"])),
                      link_pass_us=float(np.median(res["links"]) - np.median(res["plain"])))), flush=True)
# the pass alone over a 24,000-record write (2^20 pushed, the newest 24,000 survive): replay_push with and without links
data = [torch.rand((9, 1 << 20), device="cuda"), torch.rand((2, 1 << 20), device="cuda"), torch.rand(1 << 20, device="cuda"),
        torch.rand((9, 1 << 20), device="cuda")]
res = {"links": [], "plain": []}
for _ in range(args.reps):
    for mode in res:
        res[mode].append(timed(lambda: [small[mode].push(*data) for _ in range(10)], 10))
print(json.dumps(dict(case="push_2^20_into_24000", card=card, links_us=float(np.median(res["links"])), plain_us=float(np.median(res["plain"])),
                      link_pass_us=float(np.median(res["links"]) - np.median(res["plain"])))), flush=True)
