"""Every replay() kernel path against the Float64 restatement of tests/ddpg_f64.py.

replay() picks its kernels from the batch size, the population size and use_tensor_cores (csrc/ddpg.cu: update_regime,
enqueue_forward's nsplit, enqueue_phase1's bwd_split, use_fused).  Two kinds of checks:

Part A, bit for bit.  The data is built so that nothing rounds anywhere: every value that enters a tcgen05 product has its low 13
mantissa bits zero (TF32 conversion is the identity, truncating or rounding), and every fp32 sum has all its terms on a common
dyadic grid with sum |terms| below 2^22 grid units (exact in any order, under any split).  Small dyadic weights, s_min = 0 and
s_max = 1 (normalisation is the identity: 1 + 1f-8 rounds to 1), γ = 0 and zero learning rates, power-of-two B, rewards r = q_ref - δ
with dyadic δ (dq = 2δ/B), and the actor's output layer W3 = 0, b3 = 0 (actions exactly 0, tanh' exactly 1).  Pre-activations
exactly at 0 check relu'(0) = 0 on every epilogue.  Probe rows (δ = 0) carry 11-significant-bit TF32 operands into the forward
layer-2 product (layer-1 outputs and layer-2 weights): a bf16 operand there would move their q away from q_ref, and dq = 0 would no
longer hold.  The weight-gradient product h1ᵀ · dz2 only sees operands of a few significant bits (11-bit h1 values sit on δ = 0
rows, where dz2 = 0), so Part A does not tell TF32 from bf16 in it.  The dX chain into the actions is spread over about a seventh
of the layer-1 units (every lane, every column chunk, the last unit) and every k-block of layer 2, so that a dropped block, a
ragged tile or a mask off by one unit moves the actor's dW3 / db3.  The preconditions, coverage included, are asserted from the
reference's own intermediates, on every box (test_exact_data_preconditions).

Part B, realistic data.  init() weights, perturbed biases, default γ and learning rates; every gradient element of step 1 within
c · (the running bound of ddpg_f64), c = 2.  The largest err / bound of each path is printed.
"""
import functools
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ddpg_f64 as R  # noqa: E402
from ddpg_f64 import grid_units, lsb_exp, sig_bits, tf32_exact  # noqa: E402,F401

ACTOR, CRITIC, ACTOR_T, CRITIC_T = 0, 1, 2, 3
GRID_LIMIT = 2.0 ** 22
C_BOUND = 2.0


# ------------------------------------------------------------------------------------------------------------ Part A data
def _pick(rng, vals, shape, p=None):
    return rng.choice(np.asarray(vals, np.float64), size=shape, p=p)


@functools.lru_cache(maxsize=None)
def exact_case(B, l1, l2, seed):
    """weights (Flux layout Wt[in][out], float32), a minibatch and rewards on which every replay() path is exact (module doc)"""
    rng = np.random.default_rng(seed)
    probe = (np.arange(B) % 61) == 7                                    # δ = 0 rows that carry the 11-bit operands
    # ---- minibatch: states in [0, 1] on a 1/4 grid, actions in {0, ±1/2, ±1}; probe rows: zero except two probe features
    s = np.zeros((9, B))
    s[:7] = _pick(rng, [0, 0.25, 0.5, 1.0], (7, B), [0.4, 0.2, 0.2, 0.2])
    a = _pick(rng, [0, -1, -0.5, 0.5, 1], (2, B))
    s[:, probe] = 0.0
    a[:, probe] = 0.0
    s[8, probe] = rng.integers(512, 1024, probe.sum()) * 2 + 1        # 11 significant bits ...
    s[8, probe] /= 2048.0                                               # ... in (1/2, 1)
    s[7, probe] = 0.5
    # ---- critic: columns Ia carry the fine feature 8, columns Ib feature 7 (times 11-bit W2 rows); both are zero off the probe rows.
    # They stay clear of the last 8 units, which feed the actions (the backward chain's last, partial column chunk).
    perm = rng.permutation(l1 - 8)
    Ia, Ib = perm[:4], perm[4:8]
    Ic = np.setdiff1d(np.arange(l1), perm[:8])
    coarse_w = [0, 0, -1, -0.5, -0.25, 0.25, 0.5, 1]
    W1c = np.zeros((11, l1))
    W1c[np.ix_(np.arange(7), Ic)] = _pick(rng, coarse_w, (7, len(Ic)))
    W1c[8, Ia] = _pick(rng, [0.5, 1.0], len(Ia))
    W1c[7, Ib] = 1.0
    b1c = np.zeros(l1)
    b1c[Ic] = _pick(rng, [0, 0, -0.25, -3 / 16, -1 / 16, 1 / 16, 3 / 16, 0.5], len(Ic))
    # ---- the dX chain into the actions (what the backward chain kernel computes): about a seventh of the layer-1 units, the last 4
    # among them, feed each action with weight ±1; they read layer-2 units S3 (a few in every 32-unit k-block, the ragged last one
    # too) through weights ±1/4, and q reads S3 through ±1/4.  Every product of the chain has one magnitude, 2^-4/B: dA is a short
    # integer in those units, narrow enough for the actor's dW3 sum over B rows.
    act = rng.uniform(size=(2, len(Ic))) < 0.15
    act[:, -4:] = True
    for k in range(2):
        W1c[9 + k, Ic[act[k]]] = _pick(rng, [-1.0, 1.0], act[k].sum())
    A = Ic[act.any(0)]
    dens = min(1.0, 8.0 / l1)
    W2c = _pick(rng, [-0.5, -0.375, -0.25, -0.125, 0.125, 0.25, 0.375, 0.5], (l1, l2)) * (rng.uniform(size=(l1, l2)) < dens)
    fine = (rng.integers(512, 1024, (len(Ib), l2)) * 2 + 1) / 4096.0 * rng.choice([-1.0, 1.0], (len(Ib), l2))
    W2c[Ib] = np.where(W2c[Ib] != 0, fine, 0.0)
    S3 = np.unique(np.concatenate([k0 + rng.choice(min(32, l2 - k0), min(3, l2 - k0), replace=False) for k0 in range(0, l2, 32)]))
    W2c[np.ix_(A, S3)] = _pick(rng, [-0.25, 0.25], (len(A), len(S3))) * (rng.uniform(size=(len(A), len(S3))) < 0.08)
    for o in S3:                                                        # every S3 unit reaches both actions
        for k in range(2):
            W2c[rng.choice(Ic[act[k]], 2, replace=False), o] = _pick(rng, [-0.25, 0.25], 2)
    b2c = _pick(rng, [0, 0, 0, -0.125, -1 / 32, 1 / 32, 0.125], l2)
    W3c = np.zeros((l2, 1))
    W3c[S3, 0] = _pick(rng, [-0.25, 0.25], len(S3))
    b3c = np.array([0.25])
    # ---- actor: blind to the probe features; output layer zero
    W1a = np.zeros((9, l1))
    W1a[:7] = _pick(rng, [0, 0, 0, -1, 1], (7, l1))
    b1a = _pick(rng, [0, 0, -0.25, 0.25, 0.5], l1)
    W2a = _pick(rng, [-0.25, 0.25], (l1, l2)) * (rng.uniform(size=(l1, l2)) < dens / 2)
    b2a = _pick(rng, [0, -0.25, -0.5, -0.5], l2)
    actor = [(W1a, b1a), (W2a, b2a), (np.zeros((l2, 2)), np.zeros(2))]
    critic = [(W1c, b1c), (W2c, b2c), (W3c, b3c)]
    # ---- TD errors δ: zero on the probe rows, nonzero on a sparse set that touches every 32-row block
    delta = _pick(rng, [-1.0, -0.5, 0.5, 1.0], B) * ((rng.uniform(size=B) < min(1.0, 2048.0 / B)) | (np.arange(B) % 32 == 31))
    delta[probe] = 0.0
    lo, hi = np.zeros(9, np.float32), np.ones(9, np.float32)
    s32, a32 = s.astype(np.float32), a.astype(np.float32)
    q = R.critic_pass(actor, critic, critic, lo, hi, s32, a32, np.zeros(B), s32, gamma=0.0)["q"]
    r = q - delta
    assert np.array_equal(r.astype(np.float32).astype(np.float64), r)
    f32 = lambda net: [(w.astype(np.float32), b.astype(np.float32)) for w, b in net]
    return dict(B=B, l1=l1, l2=l2, actor=f32(actor), critic=f32(critic), s=s32, a=a32, r=r.astype(np.float32), delta=delta,
                probe=probe, lo=lo, hi=hi)


def f64(net):
    return [(w.astype(np.float64), b.astype(np.float64)) for w, b in net]


def exact_reference(c):
    cp = R.critic_pass(f64(c["actor"]), f64(c["critic"]), f64(c["critic"]), c["lo"], c["hi"], c["s"], c["a"], c["r"], c["s"], gamma=0.0)
    ap = R.actor_pass(f64(c["actor"]), f64(c["critic"]), c["lo"], c["hi"], c["s"])
    return cp, ap


def check_exact_preconditions(c):
    """both preconditions of Part A, from the reference's intermediates; returns a few counts for the log"""
    cp, ap = exact_reference(c)
    (W1c, b1c), (W2c, b2c), (W3c, b3c) = f64(c["critic"])
    (W1a, b1a), (W2a, b2a), (W3a, b3a) = f64(c["actor"])
    fc, bc = cp["fwd"], cp["bwd"]
    fa, fp, bp = ap["fwd_actor"], ap["fwd_critic"], ap["bwd_critic"]
    B = c["B"]
    np.testing.assert_array_equal(cp["dq"], 2.0 * c["delta"] / B)          # q == q_ref, γ = 0: dq = 2δ/B
    assert np.all(ap["api"] == 0.0)
    # 1. every tcgen05 operand is TF32-representable
    tf32_ops = {"critic h1": fc["h1"].v, "critic W2": W2c, "pi-critic h1": fp["h1"].v, "actor h1": fa["h1"].v, "actor W2": W2a,
                "critic dz2": bc["dz2"].v, "pi-critic dz2": bp["dz2"].v, "actor dz2": ap["bwd_actor"]["dz2"].v}
    for name, x in tf32_ops.items():
        assert tf32_exact(x), name
    # ... and some of them carry all 11 significant bits
    assert (sig_bits(fc["h1"].v) == 11).sum() > 0 and (sig_bits(W2c) == 11).sum() > 0 and (sig_bits(fp["h1"].v) == 11).sum() > 0
    # 2. every fp32 sum is exact in any order: sum |terms| < 2^22 units of its grid
    ones = np.ones((1, B))
    dq, dqpi, dA = cp["dq"][:, None], np.full((B, 1), -1.0 / B), ap["dA"]
    sums = {
        "critic L1": (cp["xs"], W1c, b1c), "critic L2": (fc["h1"].v, W2c, b2c), "critic L3": (fc["h2"].v, W3c, b3c),
        "pi-critic L1": (ap["xspi"], W1c, b1c), "pi-critic L2": (fp["h1"].v, W2c, b2c), "pi-critic L3": (fp["h2"].v, W3c, b3c),
        "actor L1": (ap["fwd_actor"]["x"].v, W1a, b1a), "actor L2": (fa["h1"].v, W2a, b2a), "actor L3": (fa["h2"].v, W3a, b3a),
        "critic dW3": (fc["h2"].v.T, dq, None), "critic db3": (ones, dq, None), "critic dz2": (dq, W3c.T, None),
        "critic dW2": (fc["h1"].v.T, bc["dz2"].v, None), "critic db2": (ones, bc["dz2"].v, None),
        "critic dz1": (bc["dz2"].v, W2c.T, None), "critic dW1": (cp["xs"].T, bc["dz1"].v, None), "critic db1": (ones, bc["dz1"].v, None),
        "pi-critic dz2": (dqpi, W3c.T, None), "pi-critic dz1": (bp["dz2"].v, W2c.T, None), "dA": (bp["dz1"].v, W1c[9:].T, None),
        "actor dW3": (fa["h2"].v.T, dA, None), "actor db3": (ones, dA, None),
    }
    units = {k: grid_units(*v) for k, v in sums.items()}
    for k, u in units.items():
        assert u < GRID_LIMIT, (k, u)
    # 3. what the test compares would change under the bugs it is for.  Critic: relu'(0) = 0 at pre-activations exactly 0 where the
    # upstream gradient is not, visible in the weight or bias gradient the mask feeds.
    seen = lambda X, D: bool(np.any(X.T @ D != 0) or np.any(D.sum(0) != 0))
    for z, dh, x, name in ((fc["z1"], bc["dh1"], cp["xs"], "critic z1"), (fc["z2"], bc["dh2"], fc["h1"].v, "critic z2")):
        assert seen(x, dh.v * (z.v == 0)), name
    assert (fa["z1"].v == 0).sum() > 0 and (fa["z2"].v == 0).sum() > 0
    # The dX chain through the critic (the backward chain kernel's only output, dA) is seen through the actor's dW3 = h2ᵀ dA and
    # db3: every part of its accumulation must move them.  m1 / m2: the chain's relu masks.
    h2a, W1act = fa["h2"].v, W1c[9:]
    m1, m2 = R.relu_mask(fp["z1"].v), R.relu_mask(fp["z2"].v)
    dz1p, dz2p, dh1p, dh2p = bp["dz1"].v, bp["dz2"].v, bp["dh1"].v, bp["dh2"].v
    l1, l2 = W2c.shape
    assert seen(h2a, dA) and np.all(np.abs(ap["grads"][2][0].v).max(0) > 0)                  # both actions
    for k0 in range(0, l2, 32):                                   # every 32-unit k-block of the dz2 · W2ᵀ product, the ragged last one too
        assert seen(h2a, (m1 * (dz2p[:, k0:k0 + 32] @ W2c[:, k0:k0 + 32].T)) @ W1act.T), ("k-block", k0)
    for n0 in range(0, l1, 32):                                   # every 32-unit column chunk of its output (both halves of a 2-CTA split)
        assert seen(h2a, dz1p[:, n0:n0 + 32] @ W1act[:, n0:n0 + 32].T), ("column chunk", n0)
    for lane in range(4):                                          # every lane of the float4 epilogue
        assert seen(h2a, dz1p[:, lane::4] @ W1act[:, lane::4].T), ("lane", lane)
    assert seen(h2a, dz1p[:, -1:] @ W1act[:, -1:].T)                                          # the last unit
    for lane in range(4):                                          # relu'(0) = 0 on the chain's dz1, in every lane ...
        assert seen(h2a, (dh1p * (fp["z1"].v == 0))[:, lane::4] @ W1act[:, lane::4].T), ("relu'(0) lane", lane)
    assert seen(h2a, (m1 * ((dh2p * (fp["z2"].v == 0)) @ W2c.T)) @ W1act.T)                   # ... and on its dz2
    assert np.abs(c["delta"]).sum() > 0 and np.all(np.abs(c["delta"]).reshape(-1, 32).sum(1) > 0) if B % 32 == 0 else True
    return max(units.values())


# one row per case: (id, path the selection rules send it to, B, l1, l2, use_tensor_cores, population, SHEMS_TC_CHAIN, fused, via)
PART_A = [
    ("fused", "cluster-fused kernels (one learner, fp32, B <= 256)", 128, 250, 500, 0, 1, None, True, "batch"),
    ("tiled", "tiled SIMT GEMM sequence (set_fused(False))", 128, 250, 500, 0, 1, None, False, "batch"),
    ("splitk", "large-batch SIMT with split-K over the batch (B >= 1024, fp32)", 2048, 250, 500, 0, 1, None, None, "batch"),
    ("tc_layers_512", "TF32 layer by layer: tc_gemm + l1_fwd + outer_mask + wcolsum_partial", 512, 250, 500, 1, 1, "0", None, "batch"),
    ("tc_layers_1024", "TF32 layer by layer (SHEMS_TC_CHAIN=0)", 1024, 250, 500, 1, 1, "0", None, "batch"),
    ("chain_1024", "chain kernels: 2-CTA forward, bwd_split 2 (SHEMS_TC_CHAIN=1)", 1024, 250, 500, 1, 1, "1", None, "batch"),
    ("chain_2048", "chain kernels: 2-CTA forward, bwd_split 2", 2048, 250, 500, 1, 1, None, None, "batch"),
    ("chain_8192", "chain kernels: 1-CTA three-net forward, 2-CTA TD forward, bwd_split 2 (captured graph)", 8192, 250, 500, 1, 1,
     None, None, "graph"),
    ("chain_16384", "chain kernels: 1-CTA forward, bwd_split 1", 16384, 250, 500, 1, 1, None, None, "batch"),
    ("chain_wide", "chain kernels at the widest nets they take (256/512)", 2048, 256, 512, 1, 1, None, None, "batch"),
    ("chain_partial_n", "chain kernels with partial N tiles (100/132, SHEMS_TC_CHAIN=1)", 1024, 100, 132, 1, 1, "1", None, "batch"),
    ("pop_chain", "population chain kernels, ragged tiles (64 of 128 rows per learner)", 64, 250, 500, 1, 16, None, None, "graph"),
    ("pop_layers", "population TF32 layer by layer (256 rows in all: below the population chain's 1024)", 64, 250, 500, 1, 4, None,
     None, "graph"),
]
PRECONDITION_SHAPES = sorted({(B, l1, l2, seed) for (_, _, B, l1, l2, _, P, _, _, _) in PART_A for seed in range(min(P, 3))})


@pytest.mark.parametrize("B,l1,l2,seed", PRECONDITION_SHAPES)
def test_exact_data_preconditions(B, l1, l2, seed):
    """the data Part A feeds the kernels is exact on every path: TF32 operands, fp32 sums, dq = 2δ/B (no GPU needed)"""
    worst = check_exact_preconditions(exact_case(B, l1, l2, seed))
    print("B=%d %d/%d seed %d: largest sum |terms| / grid = 2^%.1f" % (B, l1, l2, seed, np.log2(max(worst, 1.0))))


# ------------------------------------------------------------------------------------------------------------ device plumbing
@pytest.fixture
def learner_factory(monkeypatch):
    """Learner(...) with SHEMS_TC_CHAIN set (or unset) for its creation, closed at the end of the test"""
    import shems_b200 as sb
    made = []

    def make(chain, **kw):
        if chain is None:
            monkeypatch.delenv("SHEMS_TC_CHAIN", raising=False)
        else:
            monkeypatch.setenv("SHEMS_TC_CHAIN", chain)
        monkeypatch.delenv("SHEMS_DDPG_FUSED", raising=False)
        le = sb.Learner(params=sb.default_ddpg_params(**kw))
        made.append(le)
        return le

    yield make
    for le in made:
        le.close()


def dev(x):
    import torch
    return torch.as_tensor(np.ascontiguousarray(x), device="cuda")


def set_net(le, net, layers):
    for k, (w, b) in enumerate(layers):
        le.set_layer(net, k, w.reshape(-1), b)


def get_net(le, net):
    out = []
    for k in range(3):
        i, o = le.layer_shape(net, k)
        w, b = le.get_layer(net, k)
        out.append((w.reshape(i, o).astype(np.float64), b.astype(np.float64)))
    return out


def get_grads(le, net):
    out = []
    for k in range(3):
        i, o = le.layer_shape(net, k)
        w, b = le.get_grad(net, k)
        out.append((w.reshape(i, o), b))
    return out


def run_update(sb, le, cases, via):
    """one update on cases[l] for learner l: update_batch (single learner) or replay() with explicit indices (captured graph)"""
    B = cases[0]["s"].shape[1]
    if via == "batch":
        c = cases[0]
        le.update_batch(dev(c["s"]), dev(c["a"]), dev(c["r"]), dev(c["s2"]))
        return
    mems = []
    for c in cases:
        m = sb.Replay(B)
        m.push(dev(c["s"]), dev(c["a"]), dev(c["r"]), dev(c["s2"]))
        mems.append(m)
    idx = np.tile(np.arange(B, dtype=np.int32), (len(cases), 1, 1))
    le.replay(mems if len(cases) > 1 else mems[0], n_updates=1, idx=idx)
    le.sync()


# ------------------------------------------------------------------------------------------------------------ Part A
@pytest.mark.gpu
@pytest.mark.parametrize("case", PART_A, ids=[c[0] for c in PART_A])
def test_replay_path_bit_exact(learner_factory, case):
    import shems_b200 as sb
    name, path, B, l1, l2, tc, P, chain, fused, via = case
    print("\n%s: %s" % (name, path))
    le = learner_factory(chain, batch=B, l1=l1, l2=l2, use_tensor_cores=tc, population=P)
    if fused is not None:
        assert le.set_fused(fused) is fused
    cases = []
    for l in range(P):
        c = dict(exact_case(B, l1, l2, l))
        c["s2"] = c["s"]
        check_exact_preconditions(c)
        cases.append(c)
        le.select(l)
        for net, layers in ((ACTOR, c["actor"]), (CRITIC, c["critic"]), (ACTOR_T, c["actor"]), (CRITIC_T, c["critic"])):
            set_net(le, net, layers)
        le.set_norm(c["lo"], c["hi"])
        le.set_hparams(gamma=0.0, lr_critic=0.0, lr_actor=0.0)
    refs = [exact_reference(c) for c in cases]
    for step in (1, 2):   # zero learning rates: step 2 repeats step 1 on buffers step 1 left behind (accumulators need their reset)
        run_update(sb, le, cases, via)
        compare_exact(le, cases, refs, step)
    print("every gradient bit-exact, steps 1 and 2")


def compare_exact(le, cases, refs, step):
    for l, (c, (cp, ap)) in enumerate(zip(cases, refs)):
        le.select(l)
        for k, ((gw, gb), (rw, rb)) in enumerate(zip(get_grads(le, CRITIC), cp["grads"])):
            np.testing.assert_array_equal(gw, rw.v.astype(np.float32), err_msg="step %d learner %d critic dW%d" % (step, l, k + 1))
            np.testing.assert_array_equal(gb, rb.v.astype(np.float32), err_msg="step %d learner %d critic db%d" % (step, l, k + 1))
        ga = get_grads(le, ACTOR)
        np.testing.assert_array_equal(ga[2][0], ap["grads"][2][0].v.astype(np.float32), err_msg="step %d learner %d actor dW3" % (step, l))
        np.testing.assert_array_equal(ga[2][1], ap["grads"][2][1].v.astype(np.float32), err_msg="step %d learner %d actor db3" % (step, l))
        for k in (0, 1):                                                     # W3 = 0: nothing flows further down
            assert not ga[k][0].any() and not ga[k][1].any(), (step, l, k)
        np.testing.assert_array_equal(get_net(le, CRITIC)[1][0], f64(c["critic"])[1][0])   # lr_critic = 0 leaves the critic as it was
        lc, la = le.losses()
        assert lc == np.float32(cp["loss"]) and la == np.float32(ap["loss"]), (step, l, lc, cp["loss"], la, ap["loss"])


# ------------------------------------------------------------------------------------------------------------ Part B
PART_B = [
    ("tc_layers_1024", "TF32 layer by layer (SHEMS_TC_CHAIN=0)", 1024, 1, "0"),
    ("chain_1000", "chain kernels, ragged last tile (SHEMS_TC_CHAIN=1)", 1000, 1, "1"),
    ("chain_8192", "chain kernels: 1-CTA three-net forward, bwd_split 2", 8192, 1, None),
    ("pop_chain", "population chain kernels, ragged tiles", 64, 16, None),
]


def realistic_case(le, l, B, seed):
    """init() weights with perturbed biases and targets off the models, inputs as in test_update_parity_vs_oracle"""
    rng = np.random.default_rng(seed * 100 + l)
    le.select(l)
    nets = {}
    for net in (ACTOR, CRITIC):
        layers = []
        for k, (w, b) in enumerate(get_net(le, net)):
            b = rng.normal(0, 0.05, b.shape)
            layers.append((w.astype(np.float32), b.astype(np.float32)))
        set_net(le, net, layers)
        set_net(le, net + 2, [(w * np.float32(0.9), b * np.float32(1.1)) for w, b in layers])
        nets[net] = f64(layers)
        nets[net + 2] = f64([(w * np.float32(0.9), b * np.float32(1.1)) for w, b in layers])
    s_min = rng.uniform(-1, 0, 9).astype(np.float32)
    s_max = (s_min + rng.uniform(0.5, 3, 9)).astype(np.float32)
    s_max[5] = s_min[5]
    le.set_norm(s_min, s_max)
    s = rng.uniform(-1, 3, (9, B)).astype(np.float32)
    a = rng.uniform(-1, 1, (2, B)).astype(np.float32)
    r = rng.uniform(-5, 1, B).astype(np.float32)
    s2 = rng.uniform(-1, 3, (9, B)).astype(np.float32)
    s[5] = s_min[5]
    s2[5] = s_min[5]
    return dict(nets=nets, lo=s_min, hi=s_max, s=s, a=a, r=r, s2=s2)


@pytest.mark.gpu
@pytest.mark.parametrize("case", PART_B, ids=[c[0] for c in PART_B])
def test_replay_path_within_rigorous_bound(learner_factory, case):
    import shems_b200 as sb
    name, path, B, P, chain = case
    le = learner_factory(chain, batch=B, use_tensor_cores=1, population=P)
    le.init(7)
    cases = [realistic_case(le, l, B, 7) for l in range(P)]
    gamma = le.get_hparams()["gamma"]
    run_update(sb, le, cases, "batch" if P == 1 else "graph")
    worst = {}
    for l, c in enumerate(cases):
        le.select(l)
        n = c["nets"]
        cp = R.critic_pass(n[ACTOR_T], n[CRITIC], n[CRITIC_T], c["lo"], c["hi"], c["s"], c["a"], c["r"], c["s2"], gamma=gamma, track=True)
        ap = R.actor_pass(n[ACTOR], get_net(le, CRITIC), c["lo"], c["hi"], c["s"], track=True)   # through the critic the device updated
        for net, ref in ((CRITIC, cp), (ACTOR, ap)):
            for k, ((gw, gb), (rw, rb)) in enumerate(zip(get_grads(le, net), ref["grads"])):
                for got, want, tag in ((gw, rw, "dW%d" % (k + 1)), (gb, rb, "db%d" % (k + 1))):
                    err = np.abs(got.astype(np.float64) - want.v)
                    bound = C_BOUND * want.err
                    ratio = float((err / np.maximum(bound, 1e-300)).max())
                    key = ("critic " if net == CRITIC else "actor ") + tag
                    worst[key] = max(worst.get(key, 0.0), ratio)
                    assert np.all(err <= bound), (name, l, key, ratio)
    print("\n%s (%s): largest err / bound: %s" % (name, path, ", ".join("%s %.3f" % kv for kv in worst.items())))
