"""Times one ddpg_exploit (population-based training: the bottom share of every group takes over the learner state of a top learner)
at the BASELINE configs[4] shape on one GPU: 80 learners of 250/500, B = 120, tensor cores on, and two groupings of the same handle:
  * "10x8": 10 chargers x 8 learners, frac 0.25 -> 2 copies per group, 20 in all;
  * "shard": the charger runs of rank 0 of the 640-learner population on 8 GPUs (sharding.population_shard(0, 8): 64 + 16), frac 0.25
    -> 16 + 4 = 20 copies.
Two timings each, with CUDA events: back to back (--launches launches between two events; the sources may stay in the 126 MB L2
across launches) and one launch at a time after a 512 MB write that evicts L2 (median of --reps).  Beside them the byte floor:
2 x copies x ddpg_state_floats x 4 bytes.  The card's name, power limit and max SM clock are read in the same run.
usage: python tools/time_pbt.py [--launches 200] [--reps 50]   -> JSON lines"""
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
from shems_b200 import sharding  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--launches", type=int, default=200)
ap.add_argument("--reps", type=int, default=50)
args = ap.parse_args()
assert torch.cuda.is_available(), "this measurement needs a CUDA device"
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                      text=True).stdout.strip()
P = 80
le = sb.Learner(params=sb.default_ddpg_params(population=P, use_tensor_cores=1))
le.init(1)
state_bytes = 4 * int(le.lib.ddpg_state_floats(le._h))
score = torch.as_tensor(np.random.default_rng(0).normal(0, 1, P), device="cuda")
flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
_, shard_chargers, _ = sharding.population_shard(0, 8)
runs = [sum(1 for c in shard_chargers if c == x) for x in dict.fromkeys(shard_chargers)]


def events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


for name, groups in (("10x8", [8] * 10), ("shard", runs)):
    kw = dict(frac=0.25, keys=sb.Learner.HPARAMS, seed=3, round=0, groups=groups)
    parent = le.exploit(score, **kw)   # warm-up (module load)
    copies = int((parent >= 0).sum())
    torch.cuda.synchronize()
    e0, e1 = events()
    e0.record()
    for _ in range(args.launches):
        le.exploit(score, **kw)
    e1.record()
    torch.cuda.synchronize()
    b2b_us = 1e3 * e0.elapsed_time(e1) / args.launches
    cold = []
    for _ in range(args.reps):
        flush.fill_(1)
        e0, e1 = events()
        e0.record()
        le.exploit(score, **kw)
        e1.record()
        torch.cuda.synchronize()
        cold.append(1e3 * e0.elapsed_time(e1))
    moved = 2 * copies * state_bytes
    cold_us = float(np.median(cold))
    print(json.dumps(dict(case=name, card=card, learners=P, groups=groups, frac=0.25, copies=copies, state_bytes=state_bytes, bytes_moved=moved,
                          back_to_back_us=b2b_us, l2_flushed_median_us=cold_us, l2_flushed_min_us=float(np.min(cold)),
                          l2_flushed_GBps=moved / cold_us / 1e3, back_to_back_GBps=moved / b2b_us / 1e3)), flush=True)
