"""End-to-end population training (BASELINE configs[4] shape): P learners = chargers x seeds per GPU.
usage: python tools/train_population.py [--learners 80] [--envs 64] [--episodes 20] [--grid name=v1,v2 ...]
Under torch.distributed.run (one process per GPU) every rank trains its block of the 10 chargers x 64 seeds population
(sharding.population_shard; --learners is ignored then); no collective during training, rank 0 gathers the summaries.
--grid: the thesis's scalar hyper-parameter grid search (input.jl:58-100) inside the one population.  Names: lr_actor, lr_critic,
gamma, tau, noise_scale, or sigma (the exploration σ itself: the episodes then pass σ = 1 and each learner's noise_scale is its σ).
Learner g takes grid point g mod (number of points) of the cartesian product; the summary reports the eval return per grid point,
averaged over the learners (seeds, chargers) that share it."""
import argparse
import itertools
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import shems_b200 as sb  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--learners", type=int, default=80)
ap.add_argument("--envs", type=int, default=64)
ap.add_argument("--episodes", type=int, default=20)
ap.add_argument("--tc", type=int, default=1)
ap.add_argument("--eval-every", type=int, default=0)
ap.add_argument("--grid", nargs="*", default=[], metavar="NAME=V1,V2", help="per-learner hyper-parameter grid (cartesian product)")
args = ap.parse_args()
GRID_NAMES = ("lr_actor", "lr_critic", "gamma", "tau", "noise_scale", "sigma")
grid = {}
for item in args.grid:
    name, _, vals = item.partition("=")
    assert name in GRID_NAMES and vals, f"--grid {item!r}: expected NAME=V1,V2,... with NAME in {GRID_NAMES}"
    grid[name] = [float(v) for v in vals.split(",")]
assert not ("sigma" in grid and "noise_scale" in grid), "--grid: give sigma or noise_scale, not both"
points = [dict(zip(grid, combo)) for combo in itertools.product(*grid.values())] if grid else [{}]
CH = (1, 2, 3, 4, 5, 6, 7, 8, 9, 98)
rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
dist = None
torch.cuda.set_device(local)
if world > 1:
    import torch.distributed as dist
    from shems_b200 import sharding
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    gids, chargers, seeds = sharding.population_shard(rank, world)
    seeds = [1000 * g + s for g, s in zip(gids, seeds)]
else:
    chargers, seeds = [CH[(g // 64) % 10] for g in range(args.learners)], [1231 + g for g in range(args.learners)]
P = len(chargers)
learner_ids = gids if world > 1 else list(range(P))
grid_of = [g % len(points) for g in learner_ids]
hparams = {("noise_scale" if k == "sigma" else k): [points[i][k] for i in grid_of] for k in grid}
drv_kw = dict(sigma=1.0) if "sigma" in grid else {}
ser = sb.series.synth_charger98(4320, seed=98)
drv = sb.PopulationDriver(ser, chargers=chargers, seeds=seeds, n_envs=args.envs, device=local, use_tensor_cores=args.tc, hparams=hparams, **drv_kw)
t0 = time.time()
drv.populate_memory()
drv.min_max_buffer()
torch.cuda.synchronize()
t_pop = time.time() - t0
rule = drv.evaluate_rule_based()
first = drv.episode(train=False, rng_ep=999).cpu().numpy()
t1 = time.time()
t_eval = 0.0
for ep in range(1, args.episodes + 1):
    r = drv.episode(train=True, rng_ep=ep)
    if args.eval_every and ep % args.eval_every == 0:
        torch.cuda.synchronize()
        te = time.time()
        ev = drv.episode(train=False, rng_ep=999).cpu().numpy()
        t_eval += time.time() - te
        lc = [drv.learner.select(l).losses()[0] for l in (0, P - 1)]
        if rank == 0:
          print(json.dumps(dict(episode=ep, train_return=float(r.mean()), eval_return_mean=float(ev.mean()), eval_return_best=float(ev.max()),
                              eval_return_worst=float(ev.min()), beats_rule_based=int((ev > rule).sum()), loss_crit_first_last=lc)), flush=True)
torch.cuda.synchronize()
dt = time.time() - t1 - t_eval
last = drv.episode(train=False, rng_ep=999).cpu().numpy()
summary = dict(learners=P, chargers=sorted(set(chargers)), train_seconds=dt, eval_before=first.tolist(), eval_after=last.tolist(), rule=rule.tolist(),
               grid_of=grid_of)


def per_grid_point(grid_idx, after, before, rb):
    """eval return per grid point: mean over the learners of that point (its seeds and chargers), beside their rule-based return"""
    import numpy as np
    grid_idx, after, before, rb = (np.asarray(x) for x in (grid_idx, after, before, rb))
    return [dict(point=pt, learners=int((grid_idx == i).sum()), eval_return_before=float(before[grid_idx == i].mean()),
                 eval_return_after=float(after[grid_idx == i].mean()), rule_based=float(rb[grid_idx == i].mean()))
            for i, pt in enumerate(points) if (grid_idx == i).any()]


if dist is not None:
    every = [None] * world if rank == 0 else None
    dist.gather_object(summary, every, dst=0)
    if rank == 0:
        import numpy as np
        tot = sum(x["learners"] for x in every)
        tmax = max(x["train_seconds"] for x in every)
        after, before, rb, gi = (np.concatenate([x[k] for x in every]) for k in ("eval_after", "eval_before", "rule", "grid_of"))
        print(json.dumps(dict(gpus=world, learners=tot, chargers=sorted({c for x in every for c in x["chargers"]}), envs_per_learner=args.envs,
                              episodes=args.episodes, train_seconds_max_over_ranks=tmax, learner_updates_per_s=tot * args.episodes * 72 / tmax,
                              env_steps_per_s=tot * args.envs * args.episodes * 72 / tmax, eval_return_before=float(before.mean()),
                              eval_return_after=float(after.mean()), rule_based=float(rb.mean()), beats_rule_based=int((after > rb).sum()),
                              **(dict(grid=per_grid_point(gi, after, before, rb)) if grid else {}))), flush=True)
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0)
print(json.dumps(dict(learners=P, envs_per_learner=args.envs, episodes=args.episodes, populate_seconds=t_pop, train_seconds=dt,
                      vector_steps_per_s=args.episodes * 72 / dt, learner_updates_per_s=P * args.episodes * 72 / dt,
                      env_steps_per_s=P * args.envs * args.episodes * 72 / dt, eval_return_before=float(first.mean()),
                      eval_return_after=float(last.mean()), rule_based=float(rule.mean()),
                      **(dict(grid=per_grid_point(grid_of, last, first, rule)) if grid else {}))))
