"""Float64 restatement of the gradients of one replay() step (DDPG.jl:131-143), with a rigorous per-element error bound.

numpy float64 throughout; a net is [(W1, b1), (W2, b2), (W3, b3)] with W in the layout of Learner.get_layer / get_grad reshaped to
Wt[in][out] (Flux).  The formulas are those of oracle/ddpg_oracle.c and tests/test_oracle_ddpg.py:
  normalisation (s - lo) / ((hi - lo) + 1f-8) in Float32, TD target y = r + γ(1 - d) q', dq = 2(q - y)/B, the critic's backward
  pass, dqπ = -1/B, the dX chain through the critic into the action inputs times 1 - a², the actor's backward pass, both losses.
relu'(0) = 0 (Zygote's x > 0) everywhere.

critic_pass() and actor_pass() are separate: the actor's gradients are taken through the UPDATED critic (phase 2 of an update only
moves the targets), so a test can hand actor_pass() the critic the device holds after the step.  actor_out() is the forward-only
half that act() and the evaluation kernels compute: tanh(z3) of the actor on normalised states.  lsb_exp / sig_bits / tf32_exact /
grid_units state when data is exact on every path (TF32 operands, fp32 sums in any order).

track=True adds a running error bound to every gradient: each product is bounded by
  |got - ref| <= |eA|·|B| + |A|·|eB| + |eA|·|eB| + eps_K · (|A| + eA)·(|B| + eB),   eps_K = U_TF32 + K · 2^-24,
the magnitude pass (the same chain on |W|, |x| and |upstream gradient|, with the reference's relu masks) carrying the operands'
own bounds.  U_TF32 = 2^-9 covers truncating or rounding both operands of a product to TF32 (10 explicit bits); K · 2^-24 covers
fp32 accumulation of K terms in any order or split.  The same eps is used for every product, so the bound holds whichever of the
fp32 SIMT or TF32 tensor-core kernels computed it.  forward() takes per layer whether it may run on TF32 (actor_out: layer 2 only);
a layer that is fp32 on every path gets eps_K = (K + 2) · 2^-24.  A relu unit whose reference pre-activation lies within its own bound may flip
on the device: its full upstream |gradient| is added to the bound of what it feeds.
"""
import numpy as np

U_TF32 = 2.0 ** -9
U_FP32 = 2.0 ** -24
STATE = 9


def eps(K, tf32=True):
    """relative bound of one product of K terms: TF32 operands (if tf32) and fp32 accumulation in any order"""
    return (U_TF32 if tf32 else 2 * U_FP32) + K * U_FP32


def normalize(s, s_min, s_max):
    """[9][B] float32 states -> [B][9] float64 inputs, computed in Float32 as the device and the oracle do"""
    s = np.asarray(s, np.float32)
    lo, hi = np.asarray(s_min, np.float32), np.asarray(s_max, np.float32)
    den = (hi - lo) + np.float32(1e-8)
    return ((s - lo[:, None]) / den[:, None]).T.astype(np.float64)


def relu_mask(z):
    return (z > 0).astype(np.float64)


class Val:
    """a float64 value with an elementwise bound on the device's deviation from it (err is None: no bound tracked)"""

    def __init__(self, v, err=None):
        self.v, self.err = v, err


def _prod(A, B, K, track, tf32=True):
    """A @ B, and its bound when tracked (A, B: Val); tf32=False: a product computed in fp32 throughout"""
    v = A.v @ B.v
    if not track:
        return Val(v)
    aA, aB = np.abs(A.v), np.abs(B.v)
    eA = A.err if A.err is not None else np.zeros_like(aA)
    eB = B.err if B.err is not None else np.zeros_like(aB)
    if B.err is None:                     # exact operand (weights): two of the four products vanish
        return Val(v, eA @ aB + eps(K, tf32) * ((aA + eA) @ aB))
    e = eA @ aB + aA @ eB + eA @ eB + eps(K, tf32) * ((aA + eA) @ (aB + eB))
    return Val(v, e)


def _add_bias(z, b, K, track, tf32=True):
    v = z.v + b[None, :]
    if not track:
        return Val(v)
    return Val(v, z.err + eps(K, tf32) * np.abs(b)[None, :])


def _colsum(d, track):
    """sum over the batch of d [B][n] (a bias gradient)"""
    v = d.v.sum(0)
    if not track:
        return Val(v)
    B = d.v.shape[0]
    return Val(v, d.err.sum(0) + eps(B) * (np.abs(d.v) + d.err).sum(0))


def forward(net, x, track=False, tf32=(True, True, True)):
    """x: Val [B][in].  Returns the pre-activations z1, z2, z3 and activations h1, h2 (Val).
    tf32[k]: layer k + 1 may run on TF32 tensor cores (else its bound is that of fp32 arithmetic alone)."""
    (W1, b1), (W2, b2), (W3, b3) = net
    f = {"x": x}
    z1 = _add_bias(_prod(x, Val(W1), W1.shape[0], track, tf32[0]), b1, W1.shape[0], track, tf32[0])
    h1 = Val(np.where(z1.v > 0, z1.v, 0.0), z1.err)           # relu is 1-Lipschitz: the bound carries over, flipped or not
    z2 = _add_bias(_prod(h1, Val(W2), W2.shape[0], track, tf32[1]), b2, W2.shape[0], track, tf32[1])
    h2 = Val(np.where(z2.v > 0, z2.v, 0.0), z2.err)
    z3 = _add_bias(_prod(h2, Val(W3), W3.shape[0], track, tf32[2]), b3, W3.shape[0], track, tf32[2])
    f.update(z1=z1, h1=h1, z2=z2, h2=h2, z3=z3)
    return f


def _mask(dh, z, track):
    """dz = dh · relu'(z); a unit whose pre-activation lies within its bound may flip and pass (or drop) all of dh"""
    m = relu_mask(z.v)
    v = dh.v * m
    if not track:
        return Val(v), None
    flip = np.abs(z.v) <= z.err
    e = dh.err * m + flip * (np.abs(dh.v) + dh.err)
    return Val(v, e), flip


def backward(net, f, dout, want_dx=False, track=False):
    """dout: Val [B][J] = d loss / d output.  Returns {grads: [(dW1, db1), (dW2, db2), (dW3, db3)] as Val, dz2, dz1, dx, flips}."""
    (W1, b1), (W2, b2), (W3, b3) = net
    B = dout.v.shape[0]
    T = lambda a: Val(a.v.T, None if a.err is None else a.err.T)
    dW3 = _prod(T(f["h2"]), dout, B, track)
    db3 = _colsum(dout, track)
    dh2 = _prod(dout, Val(W3.T), W3.shape[1], track)
    dz2, flip2 = _mask(dh2, f["z2"], track)
    dW2 = _prod(T(f["h1"]), dz2, B, track)
    db2 = _colsum(dz2, track)
    dh1 = _prod(dz2, Val(W2.T), W2.shape[1], track)
    dz1, flip1 = _mask(dh1, f["z1"], track)
    dW1 = _prod(T(f["x"]), dz1, B, track)
    db1 = _colsum(dz1, track)
    out = {"grads": [(dW1, db1), (dW2, db2), (dW3, db3)], "dh2": dh2, "dz2": dz2, "dh1": dh1, "dz1": dz1, "flips": (flip1, flip2)}
    if want_dx:
        out["dx"] = _prod(dz1, Val(W1.T), W1.shape[1], track)
    return out


def _tanh(z, track):
    v = np.tanh(z.v)
    if not track:
        return Val(v)
    return Val(v, z.err + 4 * U_FP32)   # tanh is 1-Lipschitz; tanhf is within a few ulp of |tanh| <= 1


def actor_out(actor, s_min, s_max, obs, track=False, tf32=True):
    """tanh(z3) of `actor` on the states obs [9][n] (float32): Val [n][2], with its bound when tracked.  act() computes layers 1
    and 3 in fp32 on every path; tf32: layer 2 may run on TF32 tensor cores"""
    sn = normalize(obs, s_min, s_max)
    f = forward(actor, Val(sn, 2 * U_FP32 * np.abs(sn) if track else None), track, (False, tf32, False))
    return _tanh(f["z3"], track)


def critic_pass(actor_t, critic, critic_t, s_min, s_max, s, a, r, s2, done=None, gamma=0.99, track=False):
    """the critic half of one update on the minibatch s [9][B], a [2][B], r [B], s2 [9][B], done [B]:
    returns the critic's gradients, the loss, and the intermediates (q, y, dq, forward / backward dicts)"""
    B = s.shape[1]
    sn, s2n = normalize(s, s_min, s_max), normalize(s2, s_min, s_max)
    ex = (lambda x: 2 * U_FP32 * np.abs(x)) if track else (lambda x: None)   # the device may divide by a rounded reciprocal
    ft = forward(actor_t, Val(s2n, ex(s2n)), track)
    at = _tanh(ft["z3"], track)
    xs2 = Val(np.hstack([s2n, at.v]), np.hstack([ex(s2n), at.err]) if track else None)
    fqt = forward(critic_t, xs2, track)
    xs = np.hstack([sn, np.asarray(a, np.float64).T])
    fc = forward(critic, Val(xs, np.hstack([ex(sn), np.zeros((B, 2))]) if track else None), track)
    nd = 1.0 - (np.zeros(B) if done is None else np.asarray(done, np.float64))
    qt, q = fqt["z3"], fc["z3"]
    y = np.asarray(r, np.float64) + gamma * nd * qt.v[:, 0]
    dq = Val((2.0 * (q.v[:, 0] - y) / B)[:, None])
    if track:
        ey = gamma * nd * qt.err[:, 0] + 2 * U_FP32 * (np.abs(y) + gamma * np.abs(qt.v[:, 0]))
        dq.err = (2.0 / B * (q.err[:, 0] + ey) + 2 * U_FP32 * np.abs(dq.v[:, 0]))[:, None]
    bc = backward(critic, fc, dq, track=track)
    loss = float(np.mean((q.v[:, 0] - y) ** 2))
    return {"grads": bc["grads"], "loss": loss, "q": q.v[:, 0], "y": y, "dq": dq.v[:, 0], "fwd": fc, "bwd": bc, "xs": xs, "sn": sn}


def actor_pass(actor, critic, s_min, s_max, s, track=False):
    """the actor half: loss = -mean(critic(vcat(s_n, actor(s_n)))) through `critic` (the updated critic)"""
    B = s.shape[1]
    sn = normalize(s, s_min, s_max)
    ex = 2 * U_FP32 * np.abs(sn) if track else None
    fa = forward(actor, Val(sn, ex), track)
    api = _tanh(fa["z3"], track)
    xspi = Val(np.hstack([sn, api.v]), np.hstack([ex, api.err]) if track else None)
    fp = forward(critic, xspi, track)
    dqpi = Val(np.full((B, 1), -1.0 / B), np.zeros((B, 1)) if track else None)
    bp = backward(critic, fp, dqpi, want_dx=True, track=track)
    dxa = Val(bp["dx"].v[:, STATE:], None if not track else bp["dx"].err[:, STATE:])
    g = 1.0 - api.v ** 2
    dA = Val(dxa.v * g)
    if track:
        eg = 2 * np.abs(api.v) * api.err + api.err ** 2 + 2 * U_FP32
        dA.err = dxa.err * np.abs(g) + (np.abs(dxa.v) + dxa.err) * eg + 2 * U_FP32 * np.abs(dA.v)
    ba = backward(actor, fa, dA, track=track)
    loss = float(-np.mean(fp["z3"].v[:, 0]))
    return {"grads": ba["grads"], "loss": loss, "api": api.v, "dA": dA.v, "qpi": fp["z3"].v[:, 0], "fwd_actor": fa, "fwd_critic": fp,
            "bwd_critic": bp, "bwd_actor": ba, "xspi": xspi.v}


# ---------------------------------------------------------------------------------------------------------------- exact arithmetic
def lsb_exp(x):
    """exponent of the lowest set bit of every element (+inf for 0)"""
    x = np.asarray(x, np.float64)
    m, e = np.frexp(x)
    mi = np.abs(m * 2.0 ** 53).astype(np.int64)
    low = mi & -mi
    ctz = np.log2(np.where(low > 0, low, 1)).astype(np.int64)
    return np.where(x != 0, (e - 53 + ctz).astype(np.float64), np.inf)


def sig_bits(x):
    """significant bits of every nonzero element"""
    x = np.asarray(x, np.float64)
    _, e = np.frexp(x)
    return np.where(x != 0, e - lsb_exp(x), 0)


def tf32_exact(x):
    x = np.asarray(x, np.float64)
    f = x.astype(np.float32)
    return bool(np.all(f.astype(np.float64) == x) and np.all((f.view(np.uint32) & 0x1FFF) == 0))


def grid_units(A, Bm, bias=None, where=None):
    """max over the outputs of A @ Bm (+ bias) of sum |terms| / the grid every term lies on.

    The grid of output (m, n) is 2^g with g = min over k of lsb(A[m, k]) + lsb(Bm[k, n]) over nonzero terms.  It comes from one
    product: max_k 2^-(ga + gb) <= (sum_k 2^-p(ga + gb))^(1/p) <= K^(1/p) max_k, so floor(-log2(...)/p) is never above the true g."""
    A, Bm = np.asarray(A, np.float64), np.asarray(Bm, np.float64)
    ga, gb = lsb_exp(A), lsb_exp(Bm)
    oa = ga[np.isfinite(ga)].min() if np.isfinite(ga).any() else 0.0
    ob = gb[np.isfinite(gb)].min() if np.isfinite(gb).any() else 0.0
    rng = max(1.0, (ga[np.isfinite(ga)] - oa).max(initial=0), (gb[np.isfinite(gb)] - ob).max(initial=0))
    p = float(min(32, int(480 // rng)))
    a = np.where(np.isfinite(ga), np.exp2(p * (oa - np.where(np.isfinite(ga), ga, oa))), 0.0)
    b = np.where(np.isfinite(gb), np.exp2(p * (ob - np.where(np.isfinite(gb), gb, ob))), 0.0)
    P = a @ b
    with np.errstate(divide="ignore"):
        g = np.where(P > 0, np.floor(oa + ob - np.log2(np.where(P > 0, P, 1.0)) / p), np.inf)
    tot = np.abs(A) @ np.abs(Bm)
    if bias is not None:
        bias = np.asarray(bias, np.float64)
        g = np.minimum(g, lsb_exp(bias)[None, :])
        tot = tot + np.abs(bias)[None, :]
    assert np.all(np.isfinite(g) | (tot == 0))
    u = np.where(np.isfinite(g), tot * np.exp2(-np.where(np.isfinite(g), g, 0.0)), 0.0)
    if where is not None:
        u = u * where
    return float(u.max(initial=0.0))
