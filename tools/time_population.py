"""Times a population of independent DDPG learners (BASELINE configs[4]) advanced by one launch sequence.
usage: python tools/time_population.py [P] [n_updates] [batch] [use_tensor_cores] [mixed]
mixed: also time the same population with distinct per-learner hyper-parameters (every learner its own lr_actor, lr_critic, gamma,
tau: ddpg_set_hparams), alternating homogeneous and mixed windows, and report both."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import shems_b200 as sb  # noqa: E402

P = int(sys.argv[1]) if len(sys.argv) > 1 else 80
n_updates = int(sys.argv[2]) if len(sys.argv) > 2 else 100
B = int(sys.argv[3]) if len(sys.argv) > 3 else 120
tc = int(sys.argv[4]) if len(sys.argv) > 4 else 0
mixed = len(sys.argv) > 5 and sys.argv[5] == "mixed"
ser = sb.series.synth_charger98(4320, seed=98)
mems = []
for l in range(P):
    env = sb.Shems(72, ser, n_envs=500, env_id_base=500 * l)
    mem = sb.Replay(24_000)
    env.reset(rng=1 + l)
    env.rollout(sb.POLICY_RANDOM, 48, seed=1 + l, replay=mem, want_return=False)
    mems.append(mem)
le = sb.Learner(params=sb.default_ddpg_params(batch=B, population=P, use_tensor_cores=tc))
le.init(1)
for l in range(P):
    mn, mx = mems[l].min_max_buffer(24_000, rng_mm=l)
    le.select(l).set_norm(mn, mx)
le.replay(mems, rng_rpl=1, n_updates=10)
torch.cuda.synchronize()
base = le.get_hparams()


def set_all(mix):
    for l in range(P):
        f = 1.0 + 0.5 * (l % 4) if mix else 1.0   # four distinct tuples, cycled over the learners
        le.select(l).set_hparams(lr_actor=base["lr_actor"] * f, lr_critic=base["lr_critic"] / f, gamma=base["gamma"] - 0.01 * (f - 1.0),
                                 tau=base["tau"] * f)
    le.select(0)


res = {False: [], True: []}
for rep in range(3):
    for mix in ((False, True) if mixed else (False,)):
        if mixed:
            set_all(mix)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        le.replay(mems, rng_rpl=100 * rep, n_updates=n_updates)
        e1.record()
        torch.cuda.synchronize()
        res[mix].append(e0.elapsed_time(e1))
ms = sorted(res[False])[1]
lc, la = le.select(P - 1).losses()
out = dict(population=P, batch=B, tensor_cores=tc, n_updates=n_updates, us_per_population_update=1e3 * ms / n_updates,
           learner_updates_per_s=P * n_updates / ms * 1e3, tflops=10 * 256_500 * B * P * n_updates / ms / 1e9,
           loss_crit_last=lc, loss_act_last=la)
if mixed:
    mm = sorted(res[True])[1]
    out.update(us_per_population_update_mixed=1e3 * mm / n_updates, us_windows_homogeneous=[1e3 * x / n_updates for x in res[False]],
               us_windows_mixed=[1e3 * x / n_updates for x in res[True]])
print(json.dumps(out))
