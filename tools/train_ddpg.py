"""Vectorised DDPG training run (BASELINE configs[3] shape: tuned hyper-parameters, N parallel instances).

usage: python tools/train_ddpg.py --envs 8192 --episodes 100 --batch 1024 --updates-per-step 4
Prints one JSON line per evaluation and a final summary (env-steps/s, updates/s, returns vs the rule-based controller)."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import shems_b200 as sb  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--envs", type=int, default=8192)
ap.add_argument("--episodes", type=int, default=100)
ap.add_argument("--batch", type=int, default=1024)
ap.add_argument("--updates-per-step", type=int, default=4)
ap.add_argument("--mem", type=int, default=1 << 20)
ap.add_argument("--eval-every", type=int, default=25)
ap.add_argument("--seed", type=int, default=1231)
ap.add_argument("--sigma", type=float, default=0.1)
ap.add_argument("--tc", type=int, default=1, help="TF32 tensor cores for the 250x500 products")
ap.add_argument("--noise", default="gn", choices=["gn", "ou"])
ap.add_argument("--per", default=None, metavar="ALPHA,BETA0", help="prioritized replay, beta annealed from BETA0 to 1 over the episodes")
ap.add_argument("--nstep", type=int, default=1, help="n-step returns (1: the 1-step TD target)")
args = ap.parse_args()

train = sb.series.synth_charger98(4320, seed=98)
evals = sb.series.synth_charger98(1440, seed=99)
env = sb.Shems(72, train, n_envs=args.envs)
ev = sb.Shems(72, evals, n_envs=1024)          # evaluation: 1024 random 72-step windows of the eval series, deterministic policy
le = sb.Learner(params=sb.default_ddpg_params(batch=args.batch, use_tensor_cores=args.tc))   # γ=0.99, τ=1e-3, η=1e-4/1e-3, 250/500 (README.md:68-86)
le.init(args.seed)
drv = sb.Driver(env, ev, learner=le, mem_size=args.mem, ep_length=72, sigma=args.sigma, updates_per_step=args.updates_per_step,
                rng_run=args.seed, noise_type=args.noise, per=tuple(float(x) for x in args.per.split(",")) if args.per else None,
                nstep=args.nstep)
t0 = time.time()
drv.populate_memory()
drv.min_max_buffer()
torch.cuda.synchronize()
t_pop = time.time() - t0


def evaluate(policy):
    if policy == "rule":
        ev.reset(rng=4242)
        return float(ev.rollout(sb.POLICY_RULE, 72)["ep_return"].mean())
    r, _, _ = drv.episode(ev, train=False, num_steps=72, rng_ep=4242)
    return float(r.mean())


rule = evaluate("rule")
hist = [dict(episode=0, eval_return=evaluate("actor"), rule_based=rule)]
print(json.dumps(hist[-1]), flush=True)
t1 = time.time()
steps0 = drv.n_env_steps
for ep in range(1, args.episodes + 1):
    drv.set_beta(ep, args.episodes)
    r, _, _ = drv.episode(env, train=True, rng_ep=args.seed * 100003 + ep)
    if ep % args.eval_every == 0 or ep == args.episodes:
        lc, la = le.losses()
        hist.append(dict(episode=ep, train_return=float(r.mean()), eval_return=evaluate("actor"), rule_based=rule, loss_crit=lc, loss_act=la))
        print(json.dumps(hist[-1]), flush=True)
torch.cuda.synchronize()
dt = time.time() - t1
n_steps = drv.n_env_steps - steps0
n_upd = args.episodes * 72 * args.updates_per_step
print(json.dumps(dict(summary=True, envs=args.envs, episodes=args.episodes, batch=args.batch, updates_per_step=args.updates_per_step,
                      mem=args.mem, train_seconds=dt, populate_seconds=t_pop, env_steps_per_s=n_steps / dt, updates_per_s=n_upd / dt,
                      samples_per_s=n_upd * args.batch / dt, eval_first=hist[0]["eval_return"], eval_last=hist[-1]["eval_return"],
                      rule_based=rule)), flush=True)
