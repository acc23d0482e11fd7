"""f1/f3 of SURVEY §8: the result artefacts around the hot path, in the reference's formats.

* `write_results_csv` — the per-step 23-column tracker CSV of `write_to_results_file`
  (RL-SHEMS/src/memory_plotting_saving.jl:167-190; column order = the `results` row, shems_LU1.jl:476-478).
* `save_checkpoint` / `load_checkpoint` — the reference saves the actor only (BSON, :263-270) and can therefore not resume
  training; here the whole state goes into one .npz: the 4 nets in Flux layout, both optimisers (ADAM moments, β powers, update
  counter), normalisation constants, per-learner hyper-parameters, OU noise state, the best actors with their best_score /
  best_run (run_episodes' "temp" saveBSON, DDPG.jl:282-289), the replay memories — for every learner of a population handle.  The
  Julia shim turns the actor arrays back into a Flux Chain (same memory layout as Dense.W / Dense.b) for saveBSON.
"""
import numpy as np

from . import _lib as L

TRACE_HEADER = ["index", "c_ev", "EV_target", "EV", "Soc_ev", "rewards", "profit", "discomfort", "penalty", "PV_DE", "B_DE",
                "GR_DE", "PV_B", "PV_GR", "PV_EV", "B_EV", "GR_EV", "EX_EV", "GR_B", "B_GR", "B", "B_tar", "Soc_b"]


def write_results_csv(path, trace, instance=0):
    """trace: [T][23][N] float64 (device tensor or array) of an inference rollout -> CSV for one instance."""
    tr = trace.cpu().numpy() if hasattr(trace, "cpu") else np.asarray(trace)
    rows = tr[:, :, instance]
    with open(path, "w") as f:
        f.write(",".join(TRACE_HEADER) + "\n")
        for r in rows:
            f.write(",".join(repr(float(v)) for v in r) + "\n")
    return dict(rewards=float(rows[:, 5].sum()), profit=float(rows[:, 6].sum()), discomfort=float(rows[:, 7].sum()),
                penalty=float(rows[:, 8].sum()))  # the sums write_to_tracker_file appends (:208-210)


SUMMARY_HEADER = ["learner", "charger", "seed", "lr_actor", "lr_critic", "gamma", "tau", "noise_scale", "best_run", "best_score", "rewards",
                  "profit", "discomfort", "penalty"]


def write_population_results(out_dir, trace, chargers, seeds, best_run, best_score, hparams=None, prefix="results"):
    """A population's inference (PopulationDriver.inference, trace [T][23][P]): one results CSV per learner,
    `{prefix}_l{l}.csv` through write_results_csv, and `{prefix}_summary.csv` with a row per learner — index, charger, seed,
    hyper-parameters (hparams: one dict per learner with Learner.HPARAMS keys, or None), best_run, best_score and the four sums
    write_results_csv returns.  Returns the list of those sums."""
    import os
    os.makedirs(out_dir, exist_ok=True)
    sums = []
    with open(os.path.join(out_dir, f"{prefix}_summary.csv"), "w") as f:
        f.write(",".join(SUMMARY_HEADER) + "\n")
        for l in range(len(chargers)):
            sm = write_results_csv(os.path.join(out_dir, f"{prefix}_l{l}.csv"), trace, instance=l)
            sums.append(sm)
            hp = hparams[l] if hparams is not None else {}
            row = [l, int(chargers[l]), int(seeds[l])] + [repr(float(hp[k])) if k in hp else "" for k in SUMMARY_HEADER[3:8]]
            row += [int(best_run[l]), repr(float(best_score[l]))] + [repr(sm[k]) for k in SUMMARY_HEADER[10:]]
            f.write(",".join(str(x) for x in row) + "\n")
    return sums


NETS = ((L.NET_ACTOR, "actor"), (L.NET_CRITIC, "critic"), (L.NET_ACTOR_TARGET, "actor_target"), (L.NET_CRITIC_TARGET, "critic_target"))


def save_checkpoint(path, learner, s_min=None, s_max=None, memories=None, **scores):
    """The WHOLE learner state in one .npz, so a run can be resumed where it stopped (the reference cannot: saveBSON keeps the
    actor and the score arrays only, memory_plotting_saving.jl:263-270): for every learner l of the handle the four nets
    (Flux layout, `l{l}_actor_W1` ... — learner 0 also without the prefix, which is what the Julia shim turns into a Flux
    Chain), ADAM moments, β powers, update counter and normalisation constants (`l{l}_state`, `l{l}_opt`: ddpg_get_state),
    the hyper-parameters (`l{l}_hparams` = [lr_actor, lr_critic, gamma, tau, noise_scale] float32: ddpg_get_hparams), the best
    actors (`l{l}_actor_best_W1` ...) with `best_score` [P] / `best_run` [P] (ddpg_get_best; a score keyword of the same name
    replaces them), OUNoise.X when OU episodes ran, and — with `memories` (one Replay per learner) — the replay memories in logical order,
    with their priorities and p_max when they have them."""
    out = {}
    P = learner.population
    keep = getattr(learner, "_sel", 0)
    for l in range(P):
        if P > 1:
            learner.select(l)
        st, opt = learner.get_state()
        out[f"l{l}_state"], out[f"l{l}_opt"] = st, opt
        hp = learner.get_hparams()
        out[f"l{l}_hparams"] = np.array([hp[k] for k in learner.HPARAMS], np.float32)
        for net, name in NETS:
            for k in range(3):
                i, o = learner.layer_shape(net, k)
                w, b = learner.get_layer(net, k)
                out[f"l{l}_{name}_W{k + 1}"] = w.reshape(i, o).T.copy()  # Flux Dense.W: out×in
                out[f"l{l}_{name}_b{k + 1}"] = b
                if l == 0:
                    out[f"{name}_W{k + 1}"], out[f"{name}_b{k + 1}"] = out[f"l0_{name}_W{k + 1}"], b
        for k in range(3):
            i, o = learner.layer_shape(L.NET_ACTOR, k)
            w, b = learner.get_layer(L.NET_ACTOR_BEST, k)
            out[f"l{l}_actor_best_W{k + 1}"], out[f"l{l}_actor_best_b{k + 1}"] = w.reshape(i, o).T.copy(), b
    if P > 1:
        learner.select(keep)
    out["best_score"], out["best_run"] = learner.best()
    ou = learner.get_ou_state()
    if ou is not None:
        out["ou_x"] = ou
    out["population"] = np.int64(P)
    if memories is not None:
        mems = list(memories) if isinstance(memories, (list, tuple)) else [memories]
        for l, m in enumerate(mems):
            S, A, R, S2, D = m.get()
            out[f"mem{l}_s"], out[f"mem{l}_a"], out[f"mem{l}_r"], out[f"mem{l}_s2"], out[f"mem{l}_done"] = S, A, R, S2, D
            out[f"mem{l}_capacity"] = np.int64(m.capacity)
            if m.prioritized:   # the priorities, p_max and the ring's head (the tree's sums follow the slots' physical order)
                out[f"mem{l}_prio"], pm = m.priorities()
                out[f"mem{l}_pmax"] = np.float32(pm)
                out[f"mem{l}_head"] = np.int64(m.head)
    if s_min is not None:
        out["s_min"], out["s_max"] = np.asarray(s_min, np.float32), np.asarray(s_max, np.float32)
    for k, v in scores.items():
        out[k] = np.asarray(v)
    np.savez(path, **out)


def load_checkpoint(path, learner, memories=None):
    """Restores what save_checkpoint wrote: every learner's full state (a resumed run continues bit-identically,
    tests/test_resume_gpu.py) and, into the given EMPTY Replay objects, the replay memories.  Files holding only net
    arrays (weights-only checkpoints) restore the nets of learner 0; files without `l{l}_hparams` leave the hyper-parameters as
    they are, files without the best actors leave those (and best_score / best_run) as they are."""
    import torch
    z = np.load(path)
    P = learner.population
    if "l0_state" in z:
        assert int(z["population"]) == P, "checkpoint holds %d learners, the handle %d" % (int(z["population"]), P)
        keep = getattr(learner, "_sel", 0)
        for l in range(P):
            if P > 1:
                learner.select(l)
            learner.set_state(z[f"l{l}_state"], z[f"l{l}_opt"])
            if f"l{l}_hparams" in z:
                learner.set_hparams(**dict(zip(learner.HPARAMS, z[f"l{l}_hparams"].tolist())))
            if f"l{l}_actor_best_W1" in z:
                for k in range(3):
                    learner.set_layer(L.NET_ACTOR_BEST, k, np.ascontiguousarray(z[f"l{l}_actor_best_W{k + 1}"].T).ravel(),
                                      z[f"l{l}_actor_best_b{k + 1}"])
        if P > 1:
            learner.select(keep)
        if "l0_actor_best_W1" in z and "best_score" in z and "best_run" in z:
            learner.set_best(np.asarray(z["best_score"], np.float64).reshape(-1), np.asarray(z["best_run"]).astype(np.int32).reshape(-1))
        if "ou_x" in z:
            learner.set_ou_state(z["ou_x"])
    else:
        for net, name in NETS:
            for k in range(3):
                W = z[f"{name}_W{k + 1}"]
                learner.set_layer(net, k, np.ascontiguousarray(W.T).ravel(), z[f"{name}_b{k + 1}"])
        if "s_min" in z:
            learner.set_norm(z["s_min"], z["s_max"])
    if memories is not None:
        mems = list(memories) if isinstance(memories, (list, tuple)) else [memories]
        for l, m in enumerate(mems):
            assert len(m) == 0 and m.capacity == int(z[f"mem{l}_capacity"]), "restore into an empty memory of the saved capacity"
            dev = lambda x: torch.as_tensor(np.ascontiguousarray(x), device=m._dev)
            rec = [z[f"mem{l}_{k}"] for k in ("s", "a", "r", "s2", "done")]
            if f"mem{l}_head" in z and rec[2].size == m.capacity:
                # a full memory whose oldest record sat at slot head: the first `head` pushes only move the ring there
                head = int(z[f"mem{l}_head"])
                if head:
                    m.push(*[dev(x[..., :head]) for x in rec])
            if rec[2].size:
                m.push(*[dev(x) for x in rec])
            if f"mem{l}_prio" in z:
                m.enable_priorities()
                m.set_priorities(z[f"mem{l}_prio"], float(z[f"mem{l}_pmax"]))
    return z
