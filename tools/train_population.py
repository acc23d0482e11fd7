"""End-to-end population training (BASELINE configs[4] shape): P learners = chargers x seeds per GPU.
usage: python tools/train_population.py [--learners 80] [--envs 64] [--episodes 20] [--grid name=v1,v2 ...]
Under torch.distributed.run (one process per GPU) every rank trains its block of the 10 chargers x 64 seeds population
(sharding.population_shard; --learners is ignored then); no collective during training, rank 0 gathers the summaries.
--grid: the thesis's scalar hyper-parameter grid search (input.jl:58-100) inside the one population.  Names: lr_actor, lr_critic,
gamma, tau, noise_scale, or sigma (the exploration σ itself: the episodes then pass σ = 1 and each learner's noise_scale is its σ).
Learner g takes grid point g mod (number of points) of the cartesian product; the summary reports the eval return per grid point,
averaged over the learners (seeds, chargers) that share it.
--test-every K --test-runs R --inference-dir DIR: the reference protocol (run_episodes, DDPG.jl:244-298; driver :87-105) on a synthetic
evaluation series (1440 rows) and test series (3000 rows): every K episodes R noise-free evaluation episodes per learner from row 1,
each learner's best actor kept on the device, then inference of every best actor over the test series, one results CSV per learner
and a summary CSV in DIR.  The report adds best score, best run and test-set return per learner and per grid point.
--pbt EVERY,FRAC [--pbt-factors LO,HI] [--pbt-keys name,...] (needs --test-every): population-based training inside every run of equal
chargers (PopulationDriver.run_episodes(pbt=...)): after every EVERY-th evaluation round the worst floor(FRAC * m) learners of a run take
over the state of one of its best floor(FRAC * m) and perturb the named hyper-parameters by LO or HI.  Under torch.distributed each rank
does this over its own shard.  The report adds every learner's final hyper-parameters and how often it was replaced; the grid
table stays keyed by each learner's starting grid point."""
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
ap.add_argument("--test-every", type=int, default=0, help="evaluate every K episodes and keep each learner's best actor (run_episodes)")
ap.add_argument("--test-runs", type=int, default=100, help="evaluation episodes per learner and round")
ap.add_argument("--inference-dir", default=None, help="write the test-set inference CSVs of the best actors here (needs --test-every)")
ap.add_argument("--pbt", default=None, metavar="EVERY,FRAC", help="population-based training every EVERY evaluation rounds, share FRAC (needs --test-every)")
ap.add_argument("--per", default=None, metavar="ALPHA,BETA0", help="prioritized replay for every learner, beta annealed from BETA0 to 1")
ap.add_argument("--pbt-factors", default="0.8,1.25", metavar="LO,HI", help="perturbation factors of --pbt")
ap.add_argument("--pbt-keys", default=",".join(sb.Learner.HPARAMS), metavar="NAME,...", help="hyper-parameters --pbt perturbs")
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
assert args.inference_dir is None or args.test_every > 0, "--inference-dir runs the best actors: give --test-every K to choose them"
protocol = args.test_every > 0
assert args.pbt is None or protocol, "--pbt exploits the evaluation scores: give --test-every K"
pbt = None
if args.pbt:
    p_every, p_frac = args.pbt.split(",")
    lo, hi = (float(x) for x in args.pbt_factors.split(","))
    pbt = dict(every=int(p_every), frac=float(p_frac), factors=(lo, hi), keys=tuple(k for k in args.pbt_keys.split(",") if k), seed=rank)
if protocol:
    drv_kw.update(eval_series=sb.series.synth_charger98(1440, seed=1440), test_runs=args.test_runs)
if args.per:
    drv_kw["per"] = tuple(float(x) for x in args.per.split(","))
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
if protocol:   # run_episodes: training episodes with an evaluation round every --test-every episodes
    import numpy as np
    st = drv.run_episodes(args.episodes, test_every=args.test_every, pbt=pbt)
    torch.cuda.synchronize()
    dt = time.time() - t1
    rets, trace = drv.inference(sb.series.synth_charger98(3000, seed=3000))
    test_ret = rets.cpu().numpy()
    if args.inference_dir:
        hp_rows = [{k: v[l] for k, v in hparams.items()} for l in range(P)]
        if pbt is not None:   # the values the best actors' lineages ended with
            hp_rows = [dict(zip(sb.Learner.HPARAMS, st["hparams"][-1, l].tolist())) for l in range(P)]
        sb.tracker.write_population_results(os.path.join(args.inference_dir, f"rank{rank}"), trace, chargers, seeds, st["best_run"],
                                            st["best_score"], hparams=hp_rows)
    best = dict(best_score=st["best_score"].tolist(), best_run=[int(x) for x in st["best_run"]], test_return=test_ret.tolist(), grid_of=grid_of)
    if pbt is not None:
        best.update(hparams_final=st["hparams"][-1].tolist(), replaced=[int(x) for x in (st["parent"] >= 0).sum(axis=0)])
    if dist is not None:
        every = [None] * world if rank == 0 else None
        dist.gather_object(best, every, dst=0)
        if rank == 0:
            best = {k: [v for x in every for v in x[k]] for k in best}
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        gi, bs, tr = (np.asarray(best[k]) for k in ("grid_of", "best_score", "test_return"))
        print(json.dumps(dict(learners=len(gi), episodes=args.episodes, test_every=args.test_every, test_runs=args.test_runs, train_seconds=dt,
                              best_score=best["best_score"], best_run=best["best_run"], test_return=best["test_return"],
                              **({k: best[k] for k in ("hparams_final", "replaced")} if pbt is not None else {}),
                              pbt=pbt,
                              grid=[dict(point=pt, learners=int((gi == i).sum()), best_score=float(bs[gi == i].mean()),
                                         best_score_max=float(bs[gi == i].max()), test_return=float(tr[gi == i].mean()))
                                    for i, pt in enumerate(points) if (gi == i).any()])), flush=True)
    sys.exit(0)
for ep in range(1, args.episodes + 1):
    drv.set_beta(ep, args.episodes)
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
