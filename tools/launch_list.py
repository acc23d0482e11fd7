"""Lists the device work of one update (or act() call) per regime of the learner for one library build (SHEMS_B200_LIB): every
kernel's name, grid and block, and every memset / memcpy, from torch.profiler with CUDA activities, one profiled call per entry
after one warm-up call (graph capture, tensor maps).  Two builds that should enqueue the same work are compared with --compare.

    SHEMS_B200_LIB=old.so python tools/launch_list.py --out old.json
    python tools/launch_list.py --out new.json
    python tools/launch_list.py --compare old.json new.json

Eager calls (update_batch, the three ddpg_update_phase calls, act) keep their launch order per stream, which also shows what goes
to the side stream; graph replays are compared as multisets, since the graph's parallel branches may interleave differently from
one run to the next."""
import argparse
import collections
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def profile(fn):
    """the device work of one fn() call: [(stream ordinal, name, grid, block)] in start order"""
    import torch
    from torch.profiler import ProfilerActivity, profile as tprofile
    fn()   # warm-up: graph capture / instantiation, tensor maps, scratch allocation
    torch.cuda.synchronize()
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    work = sorted((e for e in events if e.get("cat") in ("kernel", "gpu_memset", "gpu_memcpy")), key=lambda e: e["ts"])
    streams = {}
    out = []
    for e in work:
        a = e.get("args", {})
        s = streams.setdefault(a.get("stream"), len(streams))   # streams numbered by their first piece of work
        out.append([s, e["name"], a.get("grid"), a.get("block")])
    return out


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, check=True)
        return q.stdout.strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError, IndexError):
        return "unknown"


def record():
    sys.path.insert(0, ROOT)
    import torch
    import shems_b200 as sb

    ser = sb.series.synth_charger98(4320, seed=98)
    env = sb.Shems(72, ser, n_envs=1024)
    mem = sb.Replay(1 << 16)
    env.reset(rng=1)
    env.rollout(sb.POLICY_RANDOM, 24, seed=1, replay=mem, want_return=False)
    mn, mx = mem.min_max_buffer(len(mem), rng_mm=1)
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1)

    def learner(B, tc=0, P=1, fused=True, chain=None):
        if chain is None:
            os.environ.pop("SHEMS_TC_CHAIN", None)
        else:
            os.environ["SHEMS_TC_CHAIN"] = chain
        le = sb.Learner(params=sb.default_ddpg_params(batch=B, population=P, use_tensor_cores=tc))
        if not fused:
            le.set_fused(False)
        le.init(1)
        for l in range(P):
            le.select(l).set_norm(mn, mx)
        return le.select(0)

    def rand(*shape):
        return torch.rand(shape, generator=g, device=dev, dtype=torch.float32)

    out = {}
    seeds = iter(range(10, 10_000))

    def one_learner(name, le, B, graph=True, eager=True, phases=True):
        if graph:
            out[name + " replay"] = dict(graph=True, work=profile(lambda: le.replay(mem, rng_rpl=next(seeds))))
        if eager:
            s, a, r, s2, d = rand(9, B), rand(2, B) * 2 - 1, rand(B), rand(9, B), torch.zeros(B, device=dev)
            out[name + " update_batch"] = dict(graph=False, work=profile(lambda: le.update_batch(s, a, r, s2, d)))
        if phases:
            out[name + " update_phase x3"] = dict(graph=False, work=profile(lambda: le.replay_dp(mem, rng_rpl=next(seeds))))

    def act(name, le, n, **kw):
        obs = rand(9, n)
        out[name] = dict(graph=False, work=profile(lambda: le.act(obs, sigma=0.1, rng_act=next(seeds), step=1, **kw)))

    le = learner(120)
    one_learner("B=120 fused", le, 120)
    act("act n=1 (fused act)", le, 1)
    act("act n=512 fp32", le, 512)
    ou = torch.zeros((2, 512), dtype=torch.float32, device=dev)
    obs = rand(9, 512)
    out["act_ou n=512 fp32"] = dict(graph=False, work=profile(lambda: le.act_ou(obs, ou, rng_act=next(seeds), step=1)))
    one_learner("B=120 tiled", learner(120, fused=False), 120, phases=False)
    one_learner("B=8192 fp32", learner(8192), 8192)
    one_learner("B=1024 TF32 layer-by-layer", learner(1024, tc=1), 1024)
    le = learner(8192, tc=1)
    one_learner("B=8192 TF32 chain", le, 8192)
    act("act n=512 TF32", le, 512)
    act("act n=4096 TF32", le, 4096)
    for name, P, tc in (("P=8 fp32", 8, 0), ("P=4 TF32 layer-by-layer", 4, 1), ("P=80 TF32 chain", 80, 1)):
        le = learner(120, tc=tc, P=P)
        out[name + " replay"] = dict(graph=True, work=profile(lambda: le.replay([mem] * P, rng_rpl=next(seeds))))
        if P == 80:
            obs = rand(9, 64 * P)
            out[name + " act_soa n=64"] = dict(graph=False, work=profile(lambda: le.act(obs, sigma=0.1, rng_act=next(seeds), step=1, soa=True)))
    for name, B, tc, fused in (("fused", 120, 0, True), ("tiled", 120, 0, False), ("TF32 chain", 2048, 1, True)):
        le = learner(B, tc=tc, fused=fused)
        le.dp_connect(0, 1, [le.dp_export()])
        le.dp_prepare()
        out[f"update_dp world 1 {name} B={B}"] = dict(graph=True, work=profile(lambda: le.replay_fused_dp(mem, rng_rpl=next(seeds))))
        assert le.dp_status() == 0
    os.environ.pop("SHEMS_TC_CHAIN", None)
    record_rollouts(sb, out)
    return dict(lib=os.path.basename(os.environ.get("SHEMS_B200_LIB", "libshems_b200.so")), card=card(), regimes=out)


def record_rollouts(sb, out):
    """one rollout per branch of shems_rollout's kernel choice: pair, trimmed (lean) at MINB 6 / 7 / 8 with and without a ring, and
    the general kernel with a trace, an obs trajectory, after set_state, with full records, with N not a multiple of 32 and with
    Float64 constants; two groups; every policy.  Every profiled call resets the env first (profile() calls it twice)."""
    import torch
    ser = sb.series.synth_charger98(600, seed=98)
    pair_n = 2 * 128 * 148 * 4   # the smallest launch whose paired grid fills a wave of 148 SMs x 4 CTAs

    def rollout(name, n=1024, policy=sb.POLICY_RANDOM, T=4, ring=False, rng=-1, set_state=False, groups=None, params=None, env=(), **kw):
        e = sb.Shems(64, ser, n_envs=n, groups=groups, params=params)
        mem = sb.Replay(e.n_envs * 8) if ring else None
        tape = torch.rand((T, 2, e.n_envs), device="cuda") * 2 - 1 if policy == sb.POLICY_TAPE else None
        if set_state:
            e.reset(rng=-1)
            obs, idx = e.state, e.idx

        def fn():
            if set_state:
                e.set_state(obs, idx)
            else:
                e.reset(rng=rng)
            e.rollout(policy, T, seed=1, tape=tape, tape_unscaled=True, replay=mem, **kw)

        saved = {k: os.environ.get(k) for k, _ in env}
        os.environ.update(dict(env))
        try:
            out["rollout " + name] = dict(graph=False, work=profile(fn))
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v

    for pol, pname in ((sb.POLICY_RULE, "rule"), (sb.POLICY_RANDOM, "random"), (sb.POLICY_TAPE, "tape")):
        rollout(f"{pname} pair ring", n=pair_n, policy=pol, ring=True)
        rollout(f"{pname} lean ring", policy=pol, ring=True)
        rollout(f"{pname} general trace", n=1000, policy=pol, want_trace=True)
        rollout(f"{pname} general full records", policy=pol, ring=True, env=[("SHEMS_RING_COMPACT", "0")])
    rollout("pair no ring", n=pair_n)
    rollout("pair forced, small", env=[("SHEMS_ROLLOUT_PAIR", "2")])
    rollout("pair off: lean", n=pair_n, env=[("SHEMS_ROLLOUT_PAIR", "0")])
    rollout("lockstep off: lean", n=pair_n, env=[("SHEMS_ROLLOUT_LOCKSTEP", "0")])
    rollout("lean random windows", n=pair_n, ring=True, rng=1)
    for n in (1024, 1024 * 128, 1100 * 128):   # the wave cost model picks MINB 6, 7 and 8
        rollout(f"lean no ring n={n}", n=n)
        rollout(f"general obs trajectory n={n}", n=n, want_obs=True)
    rollout("lean off: general compact", ring=True, env=[("SHEMS_ROLLOUT_LEAN", "0")])
    rollout("general compact N=1000", n=1000, ring=True)
    rollout("general after set_state", ring=True, set_state=True)
    rollout("general Float64 constants", params=sb.params_for_env(sb.ENV_LU7, 98), ring=True)
    rollout("two groups ring", groups=[(98, 512), (4, 512)], ring=True)
    rollout("two groups odd counts", groups=[(98, 33), (4, 64)], want_reward=True)


def canonical(entry):
    if entry["graph"]:   # multiset of (name, grid, block)
        return sorted(json.dumps(w[1:]) for w in entry["work"])
    per_stream = collections.defaultdict(list)
    for w in entry["work"]:
        per_stream[w[0]].append(w[1:])
    return sorted(json.dumps(seq) for seq in per_stream.values())   # each stream's sequence, whatever number the stream got


def compare(a_path, b_path):
    with open(a_path) as f:
        a = json.load(f)["regimes"]
    with open(b_path) as f:
        b = json.load(f)["regimes"]
    bad = sorted(set(a) ^ set(b))
    for k in sorted(set(a) & set(b)):
        same = canonical(a[k]) == canonical(b[k])
        print(f"{'same' if same else 'DIFFERENT':9s} {len(a[k]['work']):3d} / {len(b[k]['work']):3d}  {k}")
        if not same:
            bad.append(k)
    print("identical" if not bad else f"differ: {bad}")
    return 1 if bad else 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--compare", nargs=2)
    args = ap.parse_args()
    if args.compare:
        return compare(*args.compare)
    res = record()
    lines = [f' {json.dumps(k)}: {{"graph": {json.dumps(v["graph"])}, "work": [\n' + ",\n".join("  " + json.dumps(w) for w in v["work"]) + "]}"
             for k, v in res["regimes"].items()]   # one piece of work per line
    text = f'{{"lib": {json.dumps(res["lib"])}, "card": {json.dumps(res["card"])}, "regimes": {{\n' + ",\n".join(lines) + "}}\n"
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)
    else:
        print(text)
    return 0


if __name__ == "__main__":
    sys.exit(main())
