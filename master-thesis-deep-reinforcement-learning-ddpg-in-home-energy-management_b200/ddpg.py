"""Host-side mirror of the reference's DDPG globals (RL-SHEMS/algorithms/DDPG.jl and
src/memory_plotting_saving.jl:1-57) on top of the C ABI.

    reference (Julia global)                  here
    memory = CircularBuffer{Any}(MEM_SIZE)    Replay(capacity)
    remember(s, a, r, s′, done)               Replay.push / remember
    getData(batch; rng_dt)                    Replay.sample
    min_max_buffer(n; rng_mm)                 Replay.min_max_buffer
    actor / critic / *_target, opt_*          Learner (ddpg_create / ddpg_init / set_layer)
    normalize(s)                              fused into Learner.act / Learner.replay
    act(s_norm; train, rng_act)+scale_action  Learner.act
    replay(; rng_rpl)                         Learner.replay
    populate_memory / episode! / run_episodes / inference   Driver.*

Vectorised semantics (stated, because the reference runs 1 env × 1 learner): the N instances
of a `Shems` handle advance in lock step; one vector step pushes N transitions and is followed
by `updates_per_step` calls of replay().  With N = 1 and updates_per_step = 1 this is the
reference loop (DDPG.jl:186-242).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L
from .env import _ptr


class Replay:
    def __init__(self, capacity, device=0):
        self.lib = L.lib()
        h = C.c_void_p()
        L.check(self.lib.replay_create(int(capacity), int(device), C.byref(h)))
        self._h = h
        self.device = int(device)
        self._dev = torch.device("cuda", self.device)
        self._bind_stream()

    def _bind_stream(self):
        with torch.cuda.device(self.device):
            s = torch.cuda.current_stream().cuda_stream
        L.check(self.lib.replay_set_stream(self._h, C.c_void_p(s)))

    def close(self):
        if getattr(self, "_h", None):
            self.lib.replay_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        return int(self.lib.replay_length(self._h))

    @property
    def capacity(self):
        return int(self.lib.replay_capacity(self._h))

    @property
    def head(self):
        """physical slot of the next push"""
        return int(self.lib.replay_head(self._h))

    @property
    def series_copies(self):
        """env series the ring holds copies of (rollouts store compact records that point into them)"""
        return int(self.lib.replay_series_count(self._h))

    def push(self, s, a, r, s2, done=None):
        """remember(): s, s2 [9][n]; a [2][n] (UNSCALED action, DDPG.jl:229); r [n]; device float32 tensors."""
        n = r.numel()
        L.check(self.lib.replay_push(self._h, _ptr(s), _ptr(a), _ptr(r), _ptr(s2), _ptr(done), n))

    remember = push

    def sample(self, batch, rng_dt=0, idx=None):
        """getData(): returns (s [9][B], a [2][B], r [B], s′ [9][B], done [B]) device tensors."""
        d = self._dev
        s = torch.empty((9, batch), dtype=torch.float32, device=d)
        a = torch.empty((2, batch), dtype=torch.float32, device=d)
        r = torch.empty(batch, dtype=torch.float32, device=d)
        s2 = torch.empty((9, batch), dtype=torch.float32, device=d)
        dn = torch.empty(batch, dtype=torch.float32, device=d)
        ip = None
        if idx is not None:
            idx = np.ascontiguousarray(idx, np.int32)
            ip = idx.ctypes.data_as(L.PI)
        L.check(self.lib.replay_sample(self._h, int(batch), ip, int(rng_dt) & (2**64 - 1), _ptr(s), _ptr(a), _ptr(r), _ptr(s2), _ptr(dn)))
        return s, a, r, s2, dn

    def min_max_buffer(self, n_samples, rng_mm=0, idx=None):
        mn = np.empty(9, np.float32)
        mx = np.empty(9, np.float32)
        ip = None
        if idx is not None:
            idx = np.ascontiguousarray(idx, np.int32)
            ip = idx.ctypes.data_as(L.PI)
        L.check(self.lib.replay_minmax(self._h, int(n_samples), ip, int(rng_mm) & (2**64 - 1), mn.ctypes.data_as(L.PF), mx.ctypes.data_as(L.PF)))
        return mn, mx

    # ---- proportional prioritized replay (replay_enable_priorities): a sum tree of per-slot priorities beside the ring
    def enable_priorities(self):
        """every filled slot gets p_max (1 at first), every slot written from now on the p_max current at its write"""
        L.check(self.lib.replay_enable_priorities(self._h))
        self.prioritized = True
        return self

    prioritized = False

    def priorities(self):
        """(priorities [len] float32 in logical order, oldest first; p_max)"""
        p, pm = np.empty(len(self), np.float32), C.c_float()
        L.check(self.lib.replay_get_priorities(self._h, p.ctypes.data_as(L.PF), C.byref(pm)))
        return p, pm.value

    def set_priorities(self, prio, p_max):
        """checkpoint restore: prio [len] in logical order (finite, >= 0, not all 0), p_max > 0; the tree is recomputed"""
        p = np.ascontiguousarray(prio, np.float32)
        assert p.size == len(self)
        L.check(self.lib.replay_set_priorities(self._h, p.ctypes.data_as(L.PF), float(p_max)))

    def sample_prioritized(self, batch, seed=0, beta=0.4):
        """what update 0 of a prioritized Learner.replay(rng_rpl=seed) draws: (logical indices [B] int32, importance weights [B]
        float32), device tensors"""
        idx = torch.empty(batch, dtype=torch.int32, device=self._dev)
        w = torch.empty(batch, dtype=torch.float32, device=self._dev)
        L.check(self.lib.replay_sample_prioritized(self._h, int(batch), int(seed) & (2**64 - 1), float(beta), _ptr(idx), _ptr(w)))
        return idx, w

    # ---- n-step returns (replay_enable_successors): a successor link per slot, kept by every writer
    def enable_successors(self):
        """every record starts with no successor; every write from now on links a new record to the one it continues"""
        L.check(self.lib.replay_enable_successors(self._h))
        self.has_successors = True
        return self

    has_successors = False

    def successors(self):
        """successor of every record in logical order (oldest first): a logical index or -1, [len] int32"""
        nx = np.empty(len(self), np.int32)
        L.check(self.lib.replay_get_successors(self._h, nx.ctypes.data_as(L.PI)))
        return nx

    def set_successors(self, nx):
        """checkpoint restore: nx [len] in logical order, each -1 or in (i, len)"""
        nx = np.ascontiguousarray(nx, np.int32)
        assert nx.size == len(self)
        L.check(self.lib.replay_set_successors(self._h, nx.ctypes.data_as(L.PI)))

    def sample_nstep(self, batch, seed=0, n=3, gamma=0.99, idx=None):
        """what update 0 of an n-step Learner.replay(rng_rpl=seed) trains on (or the rows starting at the logical indices idx):
        (s [9][B], a [2][B], r [B], s' [9][B], done [B], k [B] int32) device tensors; r is the n-step return and done folds
        gamma^(k-1) in, so that gamma (1 - done) is the bootstrap factor gamma^k"""
        d = self._dev
        s = torch.empty((9, batch), dtype=torch.float32, device=d)
        a = torch.empty((2, batch), dtype=torch.float32, device=d)
        r = torch.empty(batch, dtype=torch.float32, device=d)
        s2 = torch.empty((9, batch), dtype=torch.float32, device=d)
        dn = torch.empty(batch, dtype=torch.float32, device=d)
        k = torch.empty(batch, dtype=torch.int32, device=d)
        ip = None
        if idx is not None:
            idx = np.ascontiguousarray(idx, np.int32)
            ip = idx.ctypes.data_as(L.PI)
        L.check(self.lib.replay_sample_nstep(self._h, int(batch), ip, int(seed) & (2**64 - 1), int(n), float(gamma), _ptr(s), _ptr(a), _ptr(r),
                                             _ptr(s2), _ptr(dn), _ptr(k)))
        return s, a, r, s2, dn, k

    def get(self):
        n = len(self)
        s, a, r, s2, d = (np.empty((9, n), np.float32), np.empty((2, n), np.float32), np.empty(n, np.float32),
                          np.empty((9, n), np.float32), np.empty(n, np.float32))
        L.check(self.lib.replay_get(self._h, *[x.ctypes.data_as(L.PF) for x in (s, a, r, s2, d)]))
        return s, a, r, s2, d


class Learner:
    """actor, critic, their targets and both ADAM optimisers (DDPG.jl:30-46, input.jl:126-127)."""

    def __init__(self, params=None, device=0, **kw):
        """population=P (keyword or params.population) builds P independent learners in one handle (BASELINE configs[4]: the
        reference's one-process-per-seed parallelism): `select(l)` picks the learner that get/set/losses address, batched
        arrays of act() gain a leading [P] dimension, replay() takes one Replay per learner."""
        self.lib = L.lib()
        self.p = params if params is not None else L.default_ddpg_params(**kw)
        h = C.c_void_p()
        L.check(self.lib.ddpg_create(C.byref(self.p), int(device), C.byref(h)))
        self._h = h
        self.population = int(self.lib.ddpg_population(h))
        self.device = int(device)
        self._dev = torch.device("cuda", self.device)
        self._bind_stream()

    def _bind_stream(self):
        with torch.cuda.device(self.device):
            s = torch.cuda.current_stream().cuda_stream
        L.check(self.lib.ddpg_set_stream(self._h, C.c_void_p(s)))

    def close(self):
        if getattr(self, "_h", None):
            self.lib.ddpg_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        L.check(self.lib.ddpg_sync(self._h))

    def set_fused(self, on=True):
        """ddpg_set_fused: cluster-fused small-batch replay() (True where the shape allows it) or the tiled-GEMM sequence.
        Returns the resulting state."""
        r = int(self.lib.ddpg_set_fused(self._h, int(bool(on))))
        if r < 0:
            L.check(r)
        return bool(r)

    def set_prioritized(self, alpha=0.6, beta=0.4, eps=1e-6):
        """ddpg_set_prioritized: proportional prioritized replay for every learner of the handle (alpha=None turns it off).
        Updates then need memories with priorities (Replay.enable_priorities), one per learner."""
        if alpha is None:
            L.check(self.lib.ddpg_set_prioritized(self._h, 0, 0.0, 0.0, 0.0))
        else:
            L.check(self.lib.ddpg_set_prioritized(self._h, 1, float(alpha), float(beta), float(eps)))
        return self

    def get_prioritized(self):
        """None, or {alpha, beta, eps} (float32 values)"""
        on, a, b, e = C.c_int32(), C.c_float(), C.c_float(), C.c_float()
        L.check(self.lib.ddpg_get_prioritized(self._h, C.byref(on), C.byref(a), C.byref(b), C.byref(e)))
        return dict(alpha=a.value, beta=b.value, eps=e.value) if on.value else None

    def set_nstep(self, n):
        """ddpg_set_nstep: n-step returns (1 <= n <= 16) for every learner of the handle; n > 1 needs memories with successor links
        (Replay.enable_successors), one per learner"""
        L.check(self.lib.ddpg_set_nstep(self._h, int(n)))
        return self

    def get_nstep(self):
        return int(self.lib.ddpg_get_nstep(self._h))

    def select(self, learner):
        """ddpg_select_learner: the learner of a population that set/get_layer, get_grad, set_norm and losses address."""
        L.check(self.lib.ddpg_select_learner(self._h, int(learner)))
        return self

    HPARAMS = ("lr_actor", "lr_critic", "gamma", "tau", "noise_scale")

    def set_hparams(self, **kw):
        """ddpg_set_hparams for the selected learner: any of lr_actor, lr_critic, gamma, tau, noise_scale (the others keep their
        values).  Noise is drawn with σ_eff = float32(σ × noise_scale); the new values apply from the next launch on."""
        bad = set(kw) - set(self.HPARAMS)
        assert not bad, f"unknown hyper-parameters {sorted(bad)}"
        hp = self.get_hparams()
        hp.update({k: float(v) for k, v in kw.items()})
        L.check(self.lib.ddpg_set_hparams(self._h, *[hp[k] for k in self.HPARAMS]))
        return self

    def get_hparams(self):
        """ddpg_get_hparams: {lr_actor, lr_critic, gamma, tau, noise_scale} of the selected learner (float32 values)."""
        v = [C.c_float() for _ in self.HPARAMS]
        L.check(self.lib.ddpg_get_hparams(self._h, *[C.byref(x) for x in v]))
        return {k: x.value for k, x in zip(self.HPARAMS, v)}

    def layer_shape(self, net, layer):
        S, A = self.p.state_size, self.p.action_size
        critic = net in (L.NET_CRITIC, L.NET_CRITIC_TARGET)
        dims = [(S + A if critic else S), self.p.l1, self.p.l2, (1 if critic else A)]
        return dims[layer], dims[layer + 1]

    def init(self, seed):
        L.check(self.lib.ddpg_init(self._h, int(seed) & (2**64 - 1)))

    def set_layer(self, net, layer, w=None, b=None):
        w = np.ascontiguousarray(w, np.float32) if w is not None else None
        b = np.ascontiguousarray(b, np.float32) if b is not None else None
        L.check(self.lib.ddpg_set_layer(self._h, net, layer, w.ctypes.data_as(L.PF) if w is not None else None,
                                        b.ctypes.data_as(L.PF) if b is not None else None))

    def _get(self, fn, net, layer):
        i, o = self.layer_shape(net, layer)
        w, b = np.empty(i * o, np.float32), np.empty(o, np.float32)
        L.check(fn(self._h, net, layer, w.ctypes.data_as(L.PF), b.ctypes.data_as(L.PF)))
        return w, b

    def get_layer(self, net, layer):
        """(weight, bias) in Flux layout: weight[o + out*i] (out×in column-major)."""
        return self._get(self.lib.ddpg_get_layer, net, layer)

    def get_grad(self, net, layer):
        return self._get(self.lib.ddpg_get_grad, net, layer)

    def set_norm(self, s_min, s_max):
        mn, mx = np.ascontiguousarray(s_min, np.float32), np.ascontiguousarray(s_max, np.float32)
        L.check(self.lib.ddpg_set_norm(self._h, mn.ctypes.data_as(L.PF), mx.ctypes.data_as(L.PF)))

    def act(self, obs, train=True, sigma=0.1, rng_act=0, step=0, env_id_base=0, noise=None, soa=False):
        """act(normalize(s); train) + scale_action for obs [9][n] -> (a [2][n] in [-1,1], scaled [2][n]).
        Population handles: obs [P][9][n] -> [P][2][n]; with soa=True every array is one SoA over all N = P*n instances
        (obs [9][N] = the state tensor of an environment handle, outputs [2][N] = what its step() takes)."""
        if soa:
            N = obs.shape[-1]
            n = N // self.population
            assert obs.numel() == 9 * N and n * self.population == N
            shape = (2, N)
        else:
            n = obs.shape[-1]
            shape = (2, n) if self.population == 1 else (self.population, 2, n)
            assert obs.numel() == 9 * n * self.population
        a = torch.empty(shape, dtype=torch.float32, device=self._dev)
        sc = torch.empty(shape, dtype=torch.float32, device=self._dev)
        sg = float(sigma) if (train and noise is None) else 0.0
        fn = self.lib.ddpg_act_soa if soa else self.lib.ddpg_act
        L.check(fn(self._h, _ptr(obs), n, sg, int(rng_act) & (2**64 - 1), int(step), int(env_id_base), _ptr(noise), _ptr(a), _ptr(sc)))
        return a, sc

    def act_ou(self, obs, ou_x, theta=0.15, mu=0.0, sigma=0.1, dt=1e-2, rng_act=0, step=0, env_id_base=0, z=None):
        """act() with noise_type == "ou" (DDPG.jl:49-55, :157-158): ou_x [2][n] float32 is OUNoise.X per instance, advanced in
        place; z [2][n] float64 standard normal draws or None -> Philox."""
        n = obs.shape[-1]
        shape = (2, n) if self.population == 1 else (self.population, 2, n)
        a = torch.empty(shape, dtype=torch.float32, device=self._dev)
        sc = torch.empty(shape, dtype=torch.float32, device=self._dev)
        L.check(self.lib.ddpg_act_ou(self._h, _ptr(obs), n, float(theta), float(mu), float(sigma), float(dt), _ptr(ou_x),
                                     int(rng_act) & (2**64 - 1), int(step), int(env_id_base), _ptr(z), _ptr(a), _ptr(sc)))
        return a, sc

    def set_noise(self, kind="gn", theta=0.15, mu=0.0, dt=1e-2):
        """noise_type of the native episode loop: "gn" or "ou" (OUNoise state is kept per instance inside the handle)."""
        L.check(self.lib.ddpg_set_noise(self._h, {"gn": 0, "ou": 1}[kind], float(theta), float(mu), float(dt)))

    def episode(self, env, memories, n_steps, train=True, sigma=0.1, rng_ep=0, updates_per_step=1, want_noise=False):
        """ddpg_episode: episode!(env; train, track = 0) for all instances of `env`, enqueued by one call (no host round trip per
        step).  memories: the learners' Replay objects (one for a single learner) or None when train is False.  Returns reward_eps
        [N] float64 (and, with want_noise, noise_eps [N] float32: the per-step mean(noise) summed over the episode, DDPG.jl:224)."""
        ret = torch.empty(env.n_envs, dtype=torch.float64, device=self._dev)
        nz = torch.zeros(env.n_envs, dtype=torch.float32, device=self._dev) if want_noise else None
        hs = None
        if memories is not None:
            mems = list(memories) if isinstance(memories, (list, tuple)) else [memories]
            assert len(mems) == self.population
            hs = (C.c_void_p * self.population)(*[m._h for m in mems])
        L.check(self.lib.ddpg_episode(self._h, env._h, hs, int(n_steps), 1 if train else 0, float(sigma), int(rng_ep) & (2**64 - 1),
                                      int(updates_per_step), int(env.env_id_base), _ptr(ret), _ptr(nz)))
        return (ret, nz) if want_noise else ret

    def rollout(self, env, n_steps, sigma=0.0, rng_ep=0, want_trace=False, want_actions=False):
        """ddpg_rollout: episode!(env; train = false, track) / inference(env; track = 1) for all instances of `env` by one call —
        a single persistent cluster kernel for one learner at the reference's widths.  reset! stays with the caller.
        Returns a dict: ep_return [N] float64, trace [T][23][N] float64 (want_trace), actions [T][2][N] (want_actions)."""
        n, T = env.n_envs, int(n_steps)
        out = {"ep_return": torch.empty(n, dtype=torch.float64, device=self._dev)}
        if want_trace:
            out["trace"] = torch.empty((T, 23, n), dtype=torch.float64, device=self._dev)
        if want_actions:
            out["actions"] = torch.empty((T, 2, n), dtype=torch.float32, device=self._dev)
        L.check(self.lib.ddpg_rollout(self._h, env._h, T, float(sigma), int(rng_ep) & (2**64 - 1), int(env.env_id_base),
                                      _ptr(out["ep_return"]), _ptr(out.get("trace")), _ptr(out.get("actions"))))
        return out

    def evaluate(self, env, n_steps, best=False, want_trace=False, want_actions=False):
        """ddpg_evaluate: episode!(env; train = false) / inference(env; track = 1) for EVERY learner, noise-free, by one call — the
        persistent cluster kernel with a learner dimension.  env holds N = P*n instances (learner l owns l*n .. l*n+n-1; for P > 1
        no group may split a learner); best=True runs the best-actor slots.  reset! stays with the caller.  Returns the dict of rollout()."""
        N, T = env.n_envs, int(n_steps)
        out = {"ep_return": torch.empty(N, dtype=torch.float64, device=self._dev)}
        if want_trace:
            out["trace"] = torch.empty((T, 23, N), dtype=torch.float64, device=self._dev)
        if want_actions:
            out["actions"] = torch.empty((T, 2, N), dtype=torch.float32, device=self._dev)
        L.check(self.lib.ddpg_evaluate(self._h, env._h, L.NET_ACTOR_BEST if best else L.NET_ACTOR, T, int(env.env_id_base),
                                       _ptr(out["ep_return"]), _ptr(out.get("trace")), _ptr(out.get("actions"))))
        return out

    def keep_best(self, ep_return, n, episode):
        """ddpg_keep_best: score_l = mean of ep_return[l*n .. l*n+n-1] (index order, Float64); where score_l > best_score_l (strict)
        the learner's actor goes into its best-actor slot and best_run_l = episode.  Enqueued only; returns the scores [P] (device)."""
        assert ep_return.dtype == torch.float64 and ep_return.numel() == int(n) * self.population
        score = torch.empty(self.population, dtype=torch.float64, device=self._dev)
        L.check(self.lib.ddpg_keep_best(self._h, _ptr(ep_return), int(n), int(episode), _ptr(score)))
        return score

    def best(self):
        """ddpg_get_best: (best_score [P] float64, best_run [P] int32) of every learner."""
        sc, run = np.empty(self.population, np.float64), np.empty(self.population, np.int32)
        L.check(self.lib.ddpg_get_best(self._h, sc.ctypes.data_as(L.PD), run.ctypes.data_as(L.PI)))
        return sc, run

    def set_best(self, best_score, best_run):
        """ddpg_set_best: every learner's best_score / best_run (the best-actor weights go through set_layer(NET_ACTOR_BEST, ...))."""
        sc = np.ascontiguousarray(np.broadcast_to(np.asarray(best_score, np.float64), (self.population,)))
        run = np.ascontiguousarray(np.broadcast_to(np.asarray(best_run, np.int32), (self.population,)))
        L.check(self.lib.ddpg_set_best(self._h, sc.ctypes.data_as(L.PD), run.ctypes.data_as(L.PI)))

    def exploit(self, score, frac, factors=(0.8, 1.25), keys=HPARAMS, seed=0, round=0, groups=None):
        """ddpg_exploit (population-based training): in every group the learners ranked in the bottom floor(frac * m) by `score`
        (the [P] float64 device tensor keep_best returns; NaN ranks last) take over the learner state (nets, targets, ADAM moments
        and β powers, s_min / s_max) of a learner drawn from the top floor(frac * m), and the hyper-parameters named in `keys` become
        float32(source value × factors[0] or factors[1]), γ and τ at most 1.  groups: learners per group in order (summing to P) or
        None for one group.  Enqueued only; returns parent [P] int32 (device): the source of a replaced learner, -1 otherwise."""
        assert score.dtype == torch.float64 and score.numel() == self.population and score.is_cuda and score.is_contiguous()
        bad = set(keys) - set(self.HPARAMS)
        assert not bad, f"unknown hyper-parameters {sorted(bad)}"
        p = L.DdpgExploitParams()
        p.frac, p.factor_lo, p.factor_hi = float(frac), float(factors[0]), float(factors[1])
        p.keys = sum(1 << self.HPARAMS.index(k) for k in set(keys))
        p.round, p.seed = int(round) & 0xFFFFFFFF, int(seed) & (2**64 - 1)
        if groups is not None:
            sizes = [int(x) for x in groups]
            assert len(sizes) <= L.EXPLOIT_MAX_GROUPS, f"{len(sizes)} groups, at most {L.EXPLOIT_MAX_GROUPS}"
            p.n_groups = len(sizes)
            p.group_start[:len(sizes) + 1] = np.concatenate([[0], np.cumsum(sizes)]).astype(int).tolist()
        parent = torch.empty(self.population, dtype=torch.int32, device=self._dev)
        L.check(self.lib.ddpg_exploit(self._h, _ptr(score), C.byref(p), _ptr(parent)))
        return parent

    # ---- full snapshot (nets, targets, ADAM moments, β powers, update counter, s_min/s_max): resume where the run stopped
    def get_state(self):
        n = int(self.lib.ddpg_state_floats(self._h))
        st = np.empty(n, np.float32)
        opt = np.zeros(8, np.float64)
        L.check(self.lib.ddpg_get_state(self._h, st.ctypes.data_as(L.PF), opt.ctypes.data_as(L.PD)))
        return st, opt

    def set_state(self, state, opt):
        st = np.ascontiguousarray(state, np.float32)
        op = np.ascontiguousarray(opt, np.float64)
        assert st.size == int(self.lib.ddpg_state_floats(self._h)) and op.size == 8
        L.check(self.lib.ddpg_set_state(self._h, st.ctypes.data_as(L.PF), op.ctypes.data_as(L.PD)))

    def get_ou_state(self):
        n = C.c_int64()
        L.check(self.lib.ddpg_get_ou_state(self._h, None, C.byref(n)))
        if n.value == 0:
            return None
        x = np.empty((2, n.value), np.float32)
        L.check(self.lib.ddpg_get_ou_state(self._h, x.ctypes.data_as(L.PF), C.byref(n)))
        return x

    def set_ou_state(self, x):
        x = np.ascontiguousarray(x, np.float32)
        L.check(self.lib.ddpg_set_ou_state(self._h, x.ctypes.data_as(L.PF), x.shape[-1]))

    def replay(self, memory, rng_rpl=0, n_updates=1, idx=None):
        """replay(; rng_rpl) (DDPG.jl:121-145), n_updates times back to back.  Population handles: `memory` is the list of the
        learners' Replay objects, rng_rpl an int (learner l uses rng_rpl + l) or one seed per learner, idx [P][n_updates][batch]."""
        ip = None
        if idx is not None:
            idx = np.ascontiguousarray(idx, np.int32)
            assert idx.size == n_updates * self.p.batch * self.population
            ip = idx.ctypes.data_as(L.PI)
        if self.population == 1 and not isinstance(memory, (list, tuple)):
            L.check(self.lib.ddpg_update(self._h, memory._h, int(n_updates), ip, int(rng_rpl) & (2**64 - 1)))
            return
        mems = list(memory)
        assert len(mems) == self.population
        seeds = [int(rng_rpl) + l for l in range(self.population)] if np.isscalar(rng_rpl) else [int(x) for x in rng_rpl]
        hs = (C.c_void_p * self.population)(*[m._h for m in mems])
        sd = (C.c_uint64 * self.population)(*[x & (2**64 - 1) for x in seeds])
        L.check(self.lib.ddpg_update_population(self._h, hs, int(n_updates), ip, sd))

    def replay_dp(self, memory, rng_rpl=0, dist=None, idx=None):
        """replay() for a data-parallel learner: every rank samples its own replay shard, the critic and actor gradients are
        averaged over the ranks with two NCCL all-reduces (1.03 MB in total), every rank applies the identical ADAM step."""
        world = dist.get_world_size() if (dist is not None and dist.is_initialized()) else 1
        ip = None
        if idx is not None:
            idx = np.ascontiguousarray(idx, np.int32)
            ip = idx.ctypes.data_as(L.PI)
        g = self.grad_tensor()
        nc = int(self.lib.ddpg_num_params(self._h, L.NET_CRITIC))
        seed = int(rng_rpl) & (2**64 - 1)
        L.check(self.lib.ddpg_update_phase(self._h, memory._h, 0, ip, seed, 1.0))
        if world > 1:
            dist.all_reduce(g[:nc])
        L.check(self.lib.ddpg_update_phase(self._h, memory._h, 1, None, seed, 1.0 / world))
        if world > 1:
            dist.all_reduce(g[nc:])
        L.check(self.lib.ddpg_update_phase(self._h, memory._h, 2, None, seed, 1.0 / world))

    # ---- data-parallel learner with the gradient exchange fused into the optimiser kernels (NVLink peer memory, no NCCL call)
    def dp_export(self):
        buf = C.create_string_buffer(L.DP_HANDLE_BYTES)
        L.check(self.lib.ddpg_dp_export(self._h, buf))
        return bytes(buf.raw)

    def dp_connect(self, rank, world, blobs):
        """blobs: the ranks' dp_export() results in rank order."""
        assert len(blobs) == world and all(len(b) == L.DP_HANDLE_BYTES for b in blobs)
        L.check(self.lib.ddpg_dp_connect(self._h, int(rank), int(world), C.c_char_p(b"".join(blobs))))

    def dp_connect_dist(self, dist):
        """one process per GPU: gathers the IPC handles of all ranks through torch.distributed and connects."""
        blobs = [None] * dist.get_world_size()
        dist.all_gather_object(blobs, self.dp_export())
        self.dp_connect(dist.get_rank(), dist.get_world_size(), blobs)
        self.dp_prepare()

    def dp_prepare(self, idx_ints=0):
        L.check(self.lib.ddpg_dp_prepare(self._h, int(idx_ints)))

    def replay_fused_dp(self, memory, rng_rpl=0, n_updates=1, idx=None):
        """replay() on a connected data-parallel learner (ddpg_update_dp): every rank calls it with its own replay shard."""
        ip = None
        if idx is not None:
            idx = np.ascontiguousarray(idx, np.int32)
            assert idx.size == n_updates * self.p.batch
            ip = idx.ctypes.data_as(L.PI)
        L.check(self.lib.ddpg_update_dp(self._h, memory._h, int(n_updates), ip, int(rng_rpl) & (2**64 - 1)))

    def dp_status(self):
        e = C.c_int32()
        L.check(self.lib.ddpg_dp_status(self._h, C.byref(e)))
        return e.value

    def update_batch(self, s, a, r, s2, done=None):
        L.check(self.lib.ddpg_update_batch(self._h, _ptr(s), _ptr(a), _ptr(r), _ptr(s2), _ptr(done)))

    def losses(self):
        lc, la = C.c_float(), C.c_float()
        L.check(self.lib.ddpg_get_losses(self._h, C.byref(lc), C.byref(la)))
        return lc.value, la.value

    def grad_tensor(self):
        from .env import _wrap_device
        p, n = C.c_void_p(), C.c_int64()
        L.check(self.lib.ddpg_grad_buffer(self._h, C.byref(p), C.byref(n)))
        return _wrap_device(p.value, (n.value,), torch.float32, self._dev, self)


def per_beta(beta0, episode, num_ep):
    """the importance-sampling exponent of training episode `episode` (1-based) of num_ep: linear from beta0 at the first to 1 at
    the last (Schaul et al., 2016)"""
    if episode >= num_ep:
        return 1.0
    return float(beta0) + (1.0 - float(beta0)) * (episode - 1) / (num_ep - 1)


def _per_args(per):
    """per = (alpha, beta0[, eps]) or dict(alpha, beta0, eps) -> dict, or None"""
    if per is None:
        return None
    d = dict(per) if isinstance(per, dict) else dict(zip(("alpha", "beta0", "eps"), per))
    return dict(alpha=float(d["alpha"]), beta0=float(d.get("beta0", 0.4)), eps=float(d.get("eps", 1e-6)))


class Driver:
    """DDPG_reinforce_charger_v1.jl + DDPG.jl loop glue for N lock-stepped instances.

    EP_LENGTH / NUM_EP / MEM_SIZE / noise σ follow input.jl; seeds are integers fed to Philox
    (Julia's string-concatenated MersenneTwister seeds cannot be reproduced)."""

    def __init__(self, env_train, env_eval=None, learner=None, mem_size=24_000, ep_length=72, sigma=0.1, updates_per_step=1,
                 rng_run=1231, noise_type="gn", theta=0.15, ou_dt=1e-2, native=True, per=None, nstep=1):
        """per = (alpha, beta0[, eps]) or a dict of them: proportional prioritized replay, β annealed linearly from beta0 to 1
        over the episodes of run_episodes (per_beta).  nstep > 1: n-step returns (the memory keeps successor links from its first
        write on)"""
        self.env_train, self.env_eval = env_train, env_eval
        self.learner = learner if learner is not None else Learner(device=env_train.device)
        self.memory = Replay(mem_size, device=env_train.device)
        self.mem_size, self.ep_length, self.sigma = int(mem_size), int(ep_length), float(sigma)
        self.updates_per_step = int(updates_per_step)
        self.rng_run = int(rng_run)
        self.native = bool(native)      # False: run episode! step by step from Python (reference-shaped loop; used to test the native one)
        self.s_min = self.s_max = None
        self.n_env_steps = 0
        assert noise_type in ("gn", "ou"), "parameter noise (pn) and epsilon noise (en) are out of scope (SURVEY §2)"
        self.noise_type, self.theta, self.ou_dt = noise_type, float(theta), float(ou_dt)
        self._ou_x = None  # OUNoise.X per training instance; like the reference's global `ou` it is never reset (input.jl:234)
        self.learner.set_noise(noise_type, theta=self.theta, mu=0.0, dt=self.ou_dt)
        self.per = _per_args(per)
        if self.per is not None:
            self.memory.enable_priorities()
            self.learner.set_prioritized(self.per["alpha"], self.per["beta0"], self.per["eps"])
        self.nstep = int(nstep)
        if self.nstep > 1:
            self.memory.enable_successors()
            self.learner.set_nstep(self.nstep)

    def set_beta(self, episode, num_ep):
        """prioritized replay: β of training episode `episode` of num_ep (per_beta); run_episodes calls it before every episode"""
        if self.per is not None:
            self.learner.set_prioritized(self.per["alpha"], per_beta(self.per["beta0"], episode, num_ep), self.per["eps"])

    # populate_memory(env; rng) — memory_plotting_saving.jl:9-29 (fused random-policy rollouts)
    def populate_memory(self, rng=None):
        rng = self.rng_run if rng is None else rng
        env = self.env_train
        while len(self.memory) < self.mem_size:
            env.reset(rng=rng)
            env.rollout(L.POLICY_RANDOM, self.ep_length, seed=rng, replay=self.memory, want_return=False)
            self.n_env_steps += self.ep_length * env.n_envs
            rng += 1  # `rng += 1` per episode (:26)

    # s_min, s_max = min_max_buffer(MIN_EXP_SIZE; rng_mm) — driver :30
    def min_max_buffer(self, n=None, rng_mm=None):
        n = self.mem_size if n is None else n
        self.s_min, self.s_max = self.memory.min_max_buffer(n, rng_mm=self.rng_run if rng_mm is None else rng_mm)
        self.learner.set_norm(self.s_min, self.s_max)
        return self.s_min, self.s_max

    # episode!(env; NUM_STEPS, train, track, rng_ep) — DDPG.jl:186-242
    def episode(self, env, num_steps=None, train=True, track=0, rng_ep=0):
        T = self.ep_length if num_steps is None else num_steps
        env.reset(rng=rng_ep)
        n = env.n_envs
        if track == 0 and train and self.native:
            # the whole loop below as one native call (ddpg_episode): same seeds, same kernels, no host round trip per step
            r, nz = self.learner.episode(env, self.memory, T, train=True, sigma=self.sigma, rng_ep=rng_ep,
                                         updates_per_step=self.updates_per_step, want_noise=True)
            self.n_env_steps += n * T
            return r, T, nz
        if track >= 0 and not train and self.native:
            # evaluation / DRL inference: one persistent cluster kernel for the whole episode (ddpg_rollout)
            out = self.learner.rollout(env, T, sigma=0.0, rng_ep=rng_ep, want_trace=(track != 0))
            if track == 0:
                return out["ep_return"], T, torch.zeros(n, dtype=torch.float32, device=env._torch_dev)
            return out["ep_return"], out["trace"]
        reward_eps = torch.zeros(n, dtype=torch.float64, device=env._torch_dev)
        r64 = torch.empty(n, dtype=torch.float64, device=env._torch_dev)
        noise_eps = torch.zeros(n, dtype=torch.float32, device=env._torch_dev)
        traces = []
        s_prev = torch.empty((9, n), dtype=torch.float32, device=env._torch_dev)
        for step in range(1, T + 1):
            rng_step = (rng_ep * 1000003 + step) & (2**63 - 1)
            s = env.state_tensor()
            if track < 0:
                a = env.action(track)  # DDPG.jl:210
                r, s2, tr = env.step(a, track=track, reward64_out=r64)
                traces.append(tr)
            else:
                if train and self.noise_type == "ou":
                    if self._ou_x is None or self._ou_x.shape[-1] != n:
                        self._ou_x = torch.zeros((2, n), dtype=torch.float32, device=env._torch_dev)
                    a, scaled = self.learner.act_ou(s, self._ou_x, theta=self.theta, mu=0.0, sigma=self.sigma, dt=self.ou_dt,
                                                    rng_act=rng_step, step=step, env_id_base=env.env_id_base)
                else:
                    a, scaled = self.learner.act(s, train=train, sigma=self.sigma, rng_act=rng_step, step=step, env_id_base=env.env_id_base)
                if train:
                    s_prev.copy_(s)
                if track == 0:
                    r, s2 = env.step(scaled, reward64_out=r64)
                else:
                    r, s2, tr = env.step(scaled, track=track, reward64_out=r64)
                    traces.append(tr)
            reward_eps += r64  # reward_eps += r with the Float64 env.reward (DDPG.jl:223)
            if train:
                self.memory.push(s_prev, a, r, s2)  # remember(s, a, r, s′, finished) :229
                self.learner.replay(self.memory, rng_rpl=rng_step, n_updates=self.updates_per_step)  # :231
                self.n_env_steps += n
        if track == 0:
            return reward_eps, T, noise_eps
        return reward_eps, torch.stack(traces)

    # run_episodes(env_train, env_eval, total_reward, score_mean, best_run, noise_mean, test_every, render, rng) — DDPG.jl:244-298
    def run_episodes(self, num_ep, test_every=100, test_runs=100, seed_ini=123, on_best=None, start_ep=1, state=None):
        """The training loop with the reference's bookkeeping: total_reward[i] / noise_mean[i] per training episode (:255), every
        `test_every` episodes (i % test_every == 1, :261) `test_runs` evaluation episodes of EP_LENGTH["train"] steps on env_eval
        (train = false, :266-271) -> score_mean[idx]; a new best score calls on_best(i, score) — the reference's
        saveBSON(actor, ...; idx = i, path = "temp") (:282-289) — and sets best_run = i.  The evaluation episodes run as instances
        of ONE env_eval handle (the reference runs them one after the other): test_runs is rounded up to whole batches of
        env_eval.n_envs.  `state` / `start_ep` continue a loop that was interrupted (the returned dict is that state).
        The evaluation rule is the reference's i % test_every == 1 as written, so test_every = 1 never evaluates here;
        PopulationDriver.run_episodes evaluates at i = 1, 1 + test_every, ..., which is the same rule for test_every > 1 and
        every episode for test_every = 1.
        Seeds: rng_ep = rng_run * 100003 + i, rng_test = seed_ini * 1000 + test_ep (Julia's string concatenation feeds
        MersenneTwister; here the integers key Philox streams)."""
        n = self.env_train.n_envs
        st = state if state is not None else dict(total_reward=np.zeros((num_ep, n)), noise_mean=np.zeros((num_ep, n), np.float32),
                                                  score_mean=np.zeros(-(-num_ep // test_every)), best_run=0, best_score=-100000.0)
        for i in range(start_ep, num_ep + 1):
            rng_ep = self.rng_run * 100003 + i                                        # :252
            self.set_beta(i, num_ep)
            r, _, nz = self.episode(self.env_train, train=True, rng_ep=rng_ep)        # :255
            st["total_reward"][i - 1] = r.cpu().numpy()
            st["noise_mean"][i - 1] = nz.cpu().numpy() if torch.is_tensor(nz) else nz
            if self.env_eval is not None and i % test_every == 1:                     # :261
                idx = -(-i // test_every)                                             # ceil(Int32, i / test_every) :266
                score_all, runs, test_ep = 0.0, 0, 1
                while runs < test_runs:
                    sc, _, _ = self.episode(self.env_eval, train=False, num_steps=self.ep_length, rng_ep=seed_ini * 1000 + test_ep)
                    score_all += float(sc.sum())
                    runs += self.env_eval.n_envs
                    test_ep += 1
                st["score_mean"][idx - 1] = score_all / runs                          # :273
                if st["score_mean"][idx - 1] > st["best_score"]:                     # :282-289
                    if on_best is not None:
                        on_best(i, st["score_mean"][idx - 1])
                    st["best_score"] = float(st["score_mean"][idx - 1])
                    st["best_run"] = i
        return st

    # inference(env; track) — memory_plotting_saving.jl:62-89: full-dataset deterministic rollout with the 23-column trace
    def inference(self, env, num_steps, track=1):
        if track < 0:
            env.reset(rng=-1)
            out = env.rollout(L.POLICY_RULE, num_steps, want_trace=True)
            return out["ep_return"], out["trace"]
        return self.episode(env, num_steps=num_steps, train=False, track=track, rng_ep=-1)


def push_groups(mems, s, a, r, s2, done=None):
    """remember() for a population in one launch: SoA arrays over all N = P*n_per instances, learner l's slice -> mems[l]."""
    P = len(mems)
    n_per = r.numel() // P
    hs = (C.c_void_p * P)(*[m._h for m in mems])
    L.check(mems[0].lib.replay_push_groups(hs, P, _ptr(s), _ptr(a), _ptr(r), _ptr(s2), _ptr(done), n_per))


class PopulationDriver:
    """BASELINE configs[4]: P independent DDPG runs (the reference launches one Julia process per seed / JOB_ID,
    RL-SHEMS_bs_scheduler_*.sh:73-81) advanced together.  Learner l owns n_envs environment instances (its charger's capacities,
    its own seed), a replay memory and normalisation constants.  All instances live in ONE environment handle (one group per
    run of equal chargers), so a vector step is: act (population) -> step (one launch per charger) -> remember (one launch)
    -> replay() (population).

    chargers[l] is learner l's charger id (shems_LU1.jl:47-59), equal ids must be adjacent; seeds[l] its rng_run (input.jl:136).
    hparams: per-learner hyper-parameters, a dict of lists of length P with keys from Learner.HPARAMS (lr_actor, lr_critic, gamma,
    tau, noise_scale); missing keys keep the DdpgParams values (noise_scale: 1).  Learner l explores with σ_eff = sigma × noise_scale[l],
    so a σ grid is sigma=1.0 with the grid values as noise_scale.  per = (alpha, beta0[, eps]): prioritized replay for every learner,
    β annealed from beta0 to 1 over the episodes of run_episodes, as Driver(per=...).  nstep > 1: n-step returns for every learner,
    as Driver(nstep=...).

    eval_series ([8][nrows], or [G][8][nrows] with one series per run of equal chargers) adds the reference's evaluation protocol
    (run_episodes / inference): an evaluation handle of test_runs instances per learner, one group per charger run, with
    maxsteps = nrows - 1 so that every reset! starts on row 1 (rand(1:nrows-maxsteps)).  Every learner is scored on the SAME test_runs
    starts: learner l's k-th evaluation instance starts from the draw of instance k of a one-learner evaluation handle (test_runs
    instances of its charger, env_id_base 0), as every run of the reference evaluates with the same rng."""

    def __init__(self, series, chargers, seeds, n_envs=64, mem_size=24_000, ep_length=72, sigma=0.1, device=0, use_tensor_cores=1, native=True,
                 hparams=None, eval_series=None, test_runs=100, per=None, nstep=1, **ddpg_kw):
        from .env import Shems
        assert len(chargers) == len(seeds)
        self.native = bool(native)
        self.P, self.n_envs, self.ep_length, self.sigma, self.mem_size = len(chargers), int(n_envs), int(ep_length), float(sigma), int(mem_size)
        self.seeds = [int(x) for x in seeds]
        self.chargers = [int(c) for c in chargers]
        groups = []                                      # runs of equal chargers -> instance groups
        for c in self.chargers:
            if groups and groups[-1][0] == c:
                groups[-1][1] += self.n_envs
            else:
                groups.append([c, self.n_envs])
        assert len({c for c, _ in groups}) == len(groups), "learners of the same charger must be adjacent"
        self.env = Shems(ep_length, series, device=device, env_id_base=self.seeds[0] * self.n_envs, groups=groups)
        self.N = self.env.n_envs
        self.mems = [Replay(mem_size, device=device) for _ in range(self.P)]
        self.learner = Learner(params=L.default_ddpg_params(population=self.P, use_tensor_cores=use_tensor_cores, **ddpg_kw), device=device)
        self.learner.init(self.seeds[0])            # learner l: Philox(seeds[0] + l)
        if hparams:
            for k, v in hparams.items():
                assert len(v) == self.P, f"hparams[{k!r}] has {len(v)} values for {self.P} learners"
            for l in range(self.P):
                self.learner.select(l).set_hparams(**{k: v[l] for k, v in hparams.items()})
            self.learner.select(0)
        self.per = _per_args(per)   # prioritized replay for every learner, as Driver(per=...)
        if self.per is not None:
            for m in self.mems:
                m.enable_priorities()
            self.learner.set_prioritized(self.per["alpha"], self.per["beta0"], self.per["eps"])
        self.nstep = int(nstep)     # n-step returns for every learner, as Driver(nstep=...)
        if self.nstep > 1:
            for m in self.mems:
                m.enable_successors()
            self.learner.set_nstep(self.nstep)
        self._dev = torch.device("cuda", int(device))
        self._s_prev = torch.empty((9, self.N), dtype=torch.float32, device=self._dev)
        self.n_env_steps = 0
        self._runs = [(c, k // self.n_envs) for c, k in groups]    # (charger, learners) per run of equal chargers
        self.test_runs = int(test_runs)
        self.env_eval = None
        if eval_series is not None:
            ev = np.ascontiguousarray(eval_series, np.float32)
            self.env_eval = Shems(ev.shape[-1] - 1, ev, device=device, groups=[(c, m * self.test_runs) for c, m in self._runs])
            # per charger run: the one-learner evaluation handle whose reset! draws every learner of the run starts from
            self._eval_starts, g0 = [], 0
            for g, (c, m) in enumerate(self._runs):
                ser_g = ev[g] if ev.ndim == 3 else ev
                self._eval_starts.append((g0, m, Shems(ser_g.shape[-1] - 1, ser_g, n_envs=self.test_runs, charger_id=c, device=device)))
                g0 += m * self.test_runs

    set_beta = Driver.set_beta

    def reset_eval(self, rng):
        """reset!(env_eval; rng) with the same test_runs starts for every learner: each charger run's one-learner handle is reset
        with `rng` and its states and rows are tiled over the run's learners (the population handle's own reset! sets its step and
        bounds; its draws, keyed by the global instance index, are replaced)."""
        from .env import _wrap_device
        env, R = self.env_eval, self.test_runs
        env.reset(rng=rng)
        obs = env.state_tensor()
        idx = _wrap_device(env._idx_ptr, (env.n_envs,), torch.int32, self._dev, env)
        for g0, m, one in self._eval_starts:
            one.reset(rng=rng)
            one_idx = _wrap_device(one._idx_ptr, (R,), torch.int32, self._dev, one)
            obs[:, g0:g0 + m * R].view(9, m, R).copy_(one.state_tensor().unsqueeze(1))
            idx[g0:g0 + m * R].view(m, R).copy_(one_idx.unsqueeze(0))
        return env

    def _inference_env(self, series):
        """one instance per learner on `series` (a charger run's learners share its group), reset! with rng = -1 by the caller"""
        from .env import Shems
        ser = np.ascontiguousarray(series, np.float32)
        return Shems(ser.shape[-1] - 1, ser, device=self._dev.index, groups=list(self._runs))

    def populate_memory(self):                       # memory_plotting_saving.jl:9-29 for every learner: a = 2U-1 per step, rng += 1 per episode
        rng = self.seeds[0]
        g = torch.Generator(device=self._dev).manual_seed(rng)
        while len(self.mems[-1]) < self.mem_size:
            self.env.reset(rng=rng)
            for step in range(self.ep_length):
                a = torch.rand((2, self.N), device=self._dev, generator=g) * 2.0 - 1.0
                self._s_prev.copy_(self.env.state_tensor())
                r, s2 = self.env.step((a + 1.0) * 0.5)
                push_groups(self.mems, self._s_prev, a, r, s2)
            rng += 1

    def min_max_buffer(self):                        # driver :30, per learner
        for l, mem in enumerate(self.mems):
            mn, mx = mem.min_max_buffer(self.mem_size, rng_mm=self.seeds[l])
            self.learner.select(l).set_norm(mn, mx)

    def episode(self, train=True, rng_ep=0, updates_per_step=1):
        """episode!(env; train) for every learner in lock step -> mean return per learner [P] (Float64)."""
        env = self.env
        env.reset(rng=rng_ep * 1009 + self.seeds[0])
        if self.native:
            ret = self.learner.episode(env, self.mems if train else None, self.ep_length, train=train, sigma=self.sigma, rng_ep=rng_ep,
                                       updates_per_step=updates_per_step)
            if train:
                self.n_env_steps += self.N * self.ep_length
            return ret.view(self.P, self.n_envs).mean(dim=1)
        ret = torch.zeros(self.N, dtype=torch.float64, device=self._dev)
        r64 = torch.empty(self.N, dtype=torch.float64, device=self._dev)
        for step in range(1, self.ep_length + 1):
            rng_step = (rng_ep * 1000003 + step) & (2**63 - 1)
            obs = env.state_tensor()
            a, scaled = self.learner.act(obs, train=train, sigma=self.sigma, rng_act=rng_step, step=step, env_id_base=env.env_id_base, soa=True)
            if train:
                self._s_prev.copy_(obs)
            r, s2 = env.step(scaled, reward64_out=r64)
            ret += r64                                              # reward_eps += r: the Float64 env.reward (DDPG.jl:223)
            if train:
                push_groups(self.mems, self._s_prev, a, r, s2)      # remember(s, a, r, s′, done) — the unscaled action (DDPG.jl:229)
                self.learner.replay(self.mems, rng_rpl=rng_step, n_updates=updates_per_step)
                self.n_env_steps += self.N
        return ret.view(self.P, self.n_envs).mean(dim=1)

    def evaluate_rule_based(self, rng=4242):
        """the rule-based controller (`track = -0.5`) on the same kind of windows, mean return per learner [P]"""
        self.env.reset(rng=rng)
        ret = self.env.rollout(L.POLICY_RULE, self.ep_length)["ep_return"]
        return ret.view(self.P, self.n_envs).mean(dim=1).cpu().numpy()

    # run_episodes (DDPG.jl:244-298, driver DDPG_reinforce_charger_v1.jl:87-105) for every learner at once
    def run_episodes(self, num_ep, test_every=100, seed_ini=123, on_best=None, start_ep=1, state=None, pbt=None):
        """Driver.run_episodes for the population.  Training episode i (rng_ep = seeds[0] * 100003 + i) fills total_reward[i-1] [P];
        every `test_every` episodes (i = 1, 1 + test_every, ...: the reference's i % test_every == 1, and every episode for
        test_every = 1) one evaluation round runs on the evaluation handle: ONE reset! (rng = seed_ini * 1000 + 1), one ddpg_evaluate of
        all P x test_runs instances (noise-free, ep_length steps from row 1) and one ddpg_keep_best, which forms score_mean and keeps
        each learner's best actor on the device.  The host reads the P scores only to fill score_mean[ceil(i / test_every) - 1] and to
        call on_best(l, i, score) for every learner that improved (the reference's "temp" saveBSON, :282-289).
        Every learner plays the same test_runs starts (reset_eval), so score_mean[.][l] is what learner l's actor and norm score on
        a one-learner handle with an evaluation env of test_runs instances after reset!(rng = seed_ini * 1000 + 1).
        Returns {total_reward [num_ep][P], score_mean [ceil(num_ep / test_every)][P], best_run [P], best_score [P]}.  A fresh start
        (state=None) sets best_score = -100000, best_run = 0 and zero best actors; `state` / `start_ep` continue an interrupted loop
        (its best scores are written back to the handle; restore the best actors with tracker.load_checkpoint).
        pbt = dict(every, frac, factors=(0.8, 1.25), keys=Learner.HPARAMS, seed=0) adds population-based training: after the
        keep_best of every `every`-th evaluation round r (0-based: r = every - 1, 2 every - 1, ...) one Learner.exploit with the
        runs of equal chargers as groups (an actor never moves to another household's battery) and round = r, so a resumed run
        draws the same choices.  st then also holds parent [rounds][P] int32 (-1: kept, or a round without exploit) and hparams
        [rounds][P][5] float32 (Learner.HPARAMS order), the values after the round; save them with the scores
        (tracker.save_checkpoint(**st))."""
        assert self.env_eval is not None, "run_episodes needs eval_series"
        P, te = self.P, int(test_every)
        rounds = -(-num_ep // te)
        st = state if state is not None else dict(total_reward=np.zeros((num_ep, P)), score_mean=np.zeros((rounds, P)),
                                                  best_run=np.zeros(P, np.int32), best_score=np.full(P, -100000.0))
        if pbt is not None:
            every = int(pbt["every"])
            assert every >= 1, "pbt['every'] counts evaluation rounds (>= 1)"
            pkw = dict(frac=float(pbt["frac"]), factors=tuple(pbt.get("factors", (0.8, 1.25))), keys=tuple(pbt.get("keys", Learner.HPARAMS)),
                       seed=int(pbt.get("seed", 0)), groups=[m for _, m in self._runs])
            st.setdefault("parent", np.full((rounds, P), -1, np.int32))
            st.setdefault("hparams", np.zeros((rounds, P, len(Learner.HPARAMS)), np.float32))
        self.learner.set_best(st["best_score"], st["best_run"])
        if state is None:   # no best actor left over from an earlier call on this handle
            for l in range(P):
                self.learner.select(l)
                for k in range(3):
                    i_, o_ = self.learner.layer_shape(L.NET_ACTOR, k)
                    self.learner.set_layer(L.NET_ACTOR_BEST, k, np.zeros(i_ * o_, np.float32), np.zeros(o_, np.float32))
            self.learner.select(0)
        for i in range(start_ep, num_ep + 1):
            self.set_beta(i, num_ep)
            r = self.episode(train=True, rng_ep=self.seeds[0] * 100003 + i)
            st["total_reward"][i - 1] = r.cpu().numpy()
            if (i - 1) % te == 0:
                ret = self.learner.evaluate(self.reset_eval(seed_ini * 1000 + 1), self.ep_length)["ep_return"]
                score_dev = self.learner.keep_best(ret, self.test_runs, i)
                rnd = -(-i // te) - 1
                parent = None
                if pbt is not None and (rnd + 1) % every == 0:
                    parent = self.learner.exploit(score_dev, round=rnd, **pkw)
                score = score_dev.cpu().numpy()
                st["score_mean"][rnd] = score
                for l in np.flatnonzero(score > st["best_score"]):     # the same strict rule ddpg_keep_best applied on the device
                    if on_best is not None:
                        on_best(int(l), i, float(score[l]))
                    st["best_score"][l], st["best_run"][l] = score[l], i
                if pbt is not None:
                    st["parent"][rnd] = parent.cpu().numpy() if parent is not None else -1
                    for l in range(P):
                        hp = self.learner.select(l).get_hparams()
                        st["hparams"][rnd, l] = [hp[k] for k in Learner.HPARAMS]
                    self.learner.select(0)
        return st

    # inference(env; track = 1) — memory_plotting_saving.jl:62-89, driver :95-105: one deterministic instance per learner
    def inference(self, series, num_steps=None, best=True):
        """every learner's (best) actor over `series` ([8][nrows] or one per charger run) from reset!(rng = -1), num_steps steps
        (default nrows - 1) by one ddpg_evaluate.  Returns (returns [P] float64, trace [T][23][P] float64), device tensors."""
        env = self._inference_env(series)
        T = env.nrows - 1 if num_steps is None else int(num_steps)
        env.reset(rng=-1)
        out = self.learner.evaluate(env, T, best=best, want_trace=True)
        return out["ep_return"], out["trace"]
