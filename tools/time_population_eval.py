"""Times the evaluation protocol of a population (run_episodes' evaluation round and the driver's inference, DDPG.jl:266-289,
DDPG_reinforce_charger_v1.jl:87-105) on one GPU:
  * one evaluation round at P learners x R test runs x 72 steps: ddpg_evaluate + ddpg_keep_best (the persistent cluster kernel
    with a learner dimension) against ddpg_episode(train = 0) (one population act + one step! launch pair per step), alternated,
    median of --reps;
  * inference of every learner over a 3000-row test series (2999 steps, one instance per learner) by one ddpg_evaluate;
  * the population's training vector step (ddpg_episode(train = 1), n_envs instances per learner), the yardstick of the round's cost.
The card's name and power limit are read in the same run and printed with the numbers.
usage: python tools/time_population_eval.py [--learners 80] [--test-runs 100] [--envs 64] [--reps 3]   -> JSON lines"""
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
ap.add_argument("--learners", type=int, default=80)
ap.add_argument("--test-runs", type=int, default=100)
ap.add_argument("--envs", type=int, default=64)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--train-episodes", type=int, default=3)
args = ap.parse_args()
assert torch.cuda.is_available(), "this measurement needs a CUDA device"
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                      text=True).stdout.strip()
CH = (1, 2, 3, 4, 5, 6, 7, 8, 9, 98)
P, R, T = args.learners, args.test_runs, 72
chargers, seeds = [CH[(g // 64) % 10] for g in range(P)], [1231 + g for g in range(P)]
drv = sb.PopulationDriver(sb.series.synth_charger98(4320, seed=98), chargers=chargers, seeds=seeds, n_envs=args.envs, mem_size=args.envs * T,
                          eval_series=sb.series.synth_charger98(1440, seed=1440), test_runs=R)
drv.populate_memory()
drv.min_max_buffer()
le = drv.learner


def event_ms(fn):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), out


def round_cluster():   # what run_episodes does: reset_eval (one reset per charger run, starts tiled over its learners) + evaluate + keep_best
    ret = le.evaluate(drv.reset_eval(123 * 1000 + 1), T)["ep_return"]
    return le.keep_best(ret, R, 1)


def round_pairs():    # the same starts through the population act path
    return le.episode(drv.reset_eval(123 * 1000 + 1), None, T, train=False)


round_cluster(), round_pairs()   # warm-up: module load, scratch allocation
ms = {"cluster": [], "pairs": []}
for _ in range(args.reps):
    ms["cluster"].append(event_ms(round_cluster)[0])
    ms["pairs"].append(event_ms(round_pairs)[0])
# the two paths differ by summation order (fp32 cluster kernel vs the tiled / TF32 act path): report how far the scores lie apart
sc_a = round_cluster().cpu().numpy()
sc_b = round_pairs().view(P, R).mean(dim=1).cpu().numpy()
rnd = dict(case="evaluation round", card=card, learners=P, test_runs=R, steps=T, instances=P * R,
           evaluate_keep_best_ms=float(np.median(ms["cluster"])), episode_train0_ms=float(np.median(ms["pairs"])),
           evaluate_runs_ms=ms["cluster"], episode_runs_ms=ms["pairs"], max_abs_score_diff=float(np.abs(sc_a - sc_b).max()))

env_inf = drv._inference_env(sb.series.synth_charger98(3000, seed=3000))   # what PopulationDriver.inference builds, outside the timed window


def inference():
    env_inf.reset(rng=-1)
    return le.evaluate(env_inf, 2999, want_trace=True)


inference()   # warm-up
inf = [event_ms(inference)[0] for _ in range(args.reps)]
inf_rec = dict(case="inference", card=card, learners=P, steps=2999, ms=float(np.median(inf)), runs_ms=inf,
               us_per_step=1e3 * float(np.median(inf)) / 2999)

drv.episode(train=True, rng_ep=1)    # warm-up: the update graph is captured here
tr = [event_ms(lambda i=i: drv.episode(train=True, rng_ep=2 + i))[0] for i in range(args.train_episodes)]
step_us = 1e3 * float(np.median(tr)) / T
budget_ms = 0.02 * 100 * T * step_us / 1e3
rnd.update(train_vector_step_us=step_us, train_envs_per_learner=args.envs, budget_2pct_of_100_episodes_ms=budget_ms,
           round_share_of_100_episodes=rnd["evaluate_keep_best_ms"] / (100 * T * step_us / 1e3))
print(json.dumps(rnd), flush=True)
print(json.dumps(inf_rec), flush=True)
