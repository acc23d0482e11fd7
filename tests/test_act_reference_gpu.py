"""Every act() and evaluation path against the Float64 restatement of tests/ddpg_f64.py (actor_out).

act() picks its kernels from the handle and the call (csrc/ddpg.cu: fused_act_ok, act_forward, enqueue_forward, launch_gemms):
  - the cluster-fused act kernel: one learner, use_tensor_cores = 0, a fused batch (a multiple of 8, at most FUSED_MAX_BATCH), n <= 64;
  - otherwise normalize, then layer 1 through gemm_batch (or l1_fwd_kernel once n·P >= 1024), layer 2 on TF32 tensor cores (tc_gemm)
    once n·P >= TC_MIN_ROWS = 256 on a handle with use_tensor_cores = 1 and l2 % 4 == 0, else gemm_batch, the output layer with tanh
    through gemm_skinny (gemm_batch when l2 < 32), then the noise / clamp / scale_action epilogue (Gaussian or OU).
ddpg_rollout on one learner at the fused widths and ddpg_evaluate run the persistent cluster kernel actor_rollout_kernel; ddpg_rollout
on a population or a wider net launches act + step! per step; ddpg_episode acts through act_gauss / act_ou on the environment's SoA.
Every case records its kernels once with torch.profiler and asserts the expected set.

Part A, bit for bit.  s_min = 0, s_max = 1 (normalisation is the identity: 1 + 1f-8 rounds to 1), states on a 1/4 grid, dyadic
weights with few significant bits: every layer-2 operand is TF32-representable and every fp32 sum has its terms on a common grid
below 2^22 units, so z1, z2 and z3 are exact on every path, whatever the order of the sums.  Some pre-activations are exactly 0 in
every float4 lane.  One hidden chain (state 8 -> one layer-1 unit -> one layer-2 unit -> ±1 into the two outputs, weight 16) adds
±16 to z3 on the rows with s[8] = 1: those saturate tanhf.  Every route then returns tanhf(z3) of the same float32 z3: the same
bits on every route for the same z3 (checked across all cases of a session), within 2 ulp of tanh(z3).  The first step of
ddpg_rollout / ddpg_evaluate acts on the exact start states as well: actor_rollout.cu is built with -fmad=false, ddpg.cu and
ddpg_fused.cu are not, and tanhf compiles to the same SASS either way (its FMAs are explicit), so those agree bit for bit too.

Part B, realistic data.  init() weights with random biases and the actor's W3 scaled so that z3 spreads over (about) ±7 on the
states (W3 ×40 alone leaves these states' actions in a narrow band, which hides a learner reading another learner's norm), states
from random-policy rollouts and from random_states corners, s_min / s_max from min_max_buffer widened per learner by up to half
the span (some states fall outside), Philox noise: every action element within
2 × (the ddpg_f64 running bound + the rounding of the noise add + one ulp of the re-derived noise).

Epilogues, bit for bit given the path's own noise-free output y: caller noise (past ±1 and exactly onto ±1), scale_action with
non-default bounds, the OU step with caller z over several steps; Philox noise within one ulp of the numpy Box–Muller.

Evaluation, inference and episode acts, open loop: the kernel's own actions are fed back through Shems.step, which reproduces its
states bit for bit, and every step's action is checked against actor_out on that step's state (+ the re-derived noise).
"""
import ctypes as C
import functools
import json
import os
import sys
import tempfile
import zlib

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ddpg_f64 as R  # noqa: E402
from conftest import random_states  # noqa: E402
from ddpg_f64 import grid_units, tf32_exact  # noqa: E402

ACTOR, ACTOR_BEST = 0, 4
GRID_LIMIT = 2.0 ** 22
C_BOUND = 2.0
STREAM_NOISE = 0x4E4F
E_BASE = 1000                     # env_id_base of every noisy call: noise is keyed by env_id_base + l·n + j
TANHF = {}                        # float32 z3 bits -> tanhf bits, over every route of the session


# ------------------------------------------------------------------------------------------------------------ helpers
def dev(x):
    import torch
    return torch.as_tensor(np.ascontiguousarray(x), device="cuda")


def host(t):
    return t.detach().cpu().numpy()


def f64(net):
    return [(w.astype(np.float64), b.astype(np.float64)) for w, b in net]


def set_net(le, net, layers):
    for k, (w, b) in enumerate(layers):
        le.set_layer(net, k, np.asarray(w, np.float32).reshape(-1), np.asarray(b, np.float32))


def get_net(le, net=ACTOR):
    out = []
    for k in range(3):
        i, o = le.layer_shape(net, k)
        w, b = le.get_layer(net, k)
        out.append((w.reshape(i, o).copy(), b.copy()))
    return out


def _short(name):
    """kernel name without 'void', namespace, arguments and template arguments (gemm_batch keeps its tile)"""
    name = name.replace("(anonymous namespace)::", "").split("(")[0].replace("void ", "").strip()
    base, _, targs = name.partition("<")
    return base + ("<" + targs.replace(" ", "") if base == "gemm_batch_kernel" else "")


def kernels(fn):
    """(fn()'s result, the set of kernels it launched), from torch.profiler with CUDA activities"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    return out, {_short(e["name"]) for e in events if e.get("cat") == "kernel"}


def ulp_below(x):
    """the float32 ulp just below |x| (the ulp of a float32 value in [2^e, 2^(e+1)) that rounds to |x|)"""
    return np.spacing(np.nextafter(np.abs(np.asarray(x, np.float32)), np.float32(0))).astype(np.float64)


def scale_action(a, lo, hi):
    """Float32.(LO .+ (a .+ 1.0) .* 0.5 .* (HI .- LO)) in Float64, HI - LO in Float32"""
    sp = (np.float32(hi) - np.float32(lo)).astype(np.float64)
    return (np.float64(np.float32(lo)) + (a.astype(np.float64) + 1.0) * 0.5 * sp).astype(np.float32)


def rng_step(seed, step):
    return (seed * 1000003 + step) & (2 ** 63 - 1)


@functools.lru_cache(maxsize=None)
def _oracle_lib():
    from oracle import oracle as O
    O.build()
    lib = O.lib()
    lib.oracle_u53.restype = C.c_double
    lib.oracle_u53.argtypes = [C.c_uint32, C.c_uint32]
    lib.oracle_philox.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32)]
    return lib


def standard_normals(seed, ids, step):
    """(rad·cos 2πu2, rad·sin 2πu2) [2][len(ids)] float64 from Philox(seed, id, step, STREAM_NOISE), u1 = 1 - u53, u2 = u53"""
    lib = _oracle_lib()
    w = (C.c_uint32 * 4)()
    z = np.empty((2, len(ids)))
    for i, e in enumerate(ids):
        lib.oracle_philox(int(seed), int(e), int(step), STREAM_NOISE, w)
        u1, u2 = 1.0 - lib.oracle_u53(w[0], w[1]), lib.oracle_u53(w[2], w[3])
        rad = np.sqrt(-2.0 * np.log(u1))
        z[0, i], z[1, i] = rad * np.cos(2 * np.pi * u2), rad * np.sin(2 * np.pi * u2)
    return z


def gauss_noise(seed, ids, step, sigma_eff):
    """Float32(σ_eff · z): the act epilogue's noise, re-derived"""
    return (np.float64(np.float32(sigma_eff)) * standard_normals(seed, ids, step)).astype(np.float32)


def sigma_eff(sigma, noise_scale):
    return np.float32(np.float32(sigma) * np.float32(noise_scale))


def noisy_interval(y, nz):
    """clamp(RN32(y + nz'), -1, 1) for nz' one float32 ulp either side of nz: the range a noise within one ulp can give"""
    y, nz = np.asarray(y, np.float32), np.asarray(nz, np.float32)
    lo = np.clip(y + np.nextafter(nz, np.float32(-np.inf)), -1, 1)
    hi = np.clip(y + np.nextafter(nz, np.float32(np.inf)), -1, 1)
    return lo, hi


def check_bounded(a_dev, y, nz, tag):
    """a_dev [n][2] against clamp(y.v + nz) [n][2]: within C_BOUND × (y's bound + the noise add's rounding + an ulp of the noise)"""
    nz = np.zeros_like(y.v) if nz is None else np.asarray(nz, np.float64)
    s = y.v + nz
    ref = np.clip(s, -1, 1)
    bound = y.err + R.U_FP32 * np.abs(s) + np.spacing(np.abs(nz.astype(np.float32))).astype(np.float64) * (nz != 0)
    err = np.abs(np.asarray(a_dev, np.float64) - ref)
    ratio = float((err / np.maximum(C_BOUND * bound, 1e-300)).max())
    assert np.all(err <= C_BOUND * bound), (tag, ratio, np.unravel_index(np.argmax(err / bound), err.shape))
    return ratio


def record_tanhf(z3, y, tag):
    """y (device) = tanhf(z3) for z3 exact: the same bits as every other route gave the same z3, within 2 ulp of tanh(z3)"""
    z3 = np.asarray(z3, np.float64)
    z32 = z3.astype(np.float32)
    assert np.array_equal(z32.astype(np.float64), z3), tag
    y = np.asarray(y, np.float32)
    ref = np.tanh(z3)
    assert np.all(np.abs(y.astype(np.float64) - ref) <= 2 * ulp_below(ref)), (tag, float(np.abs(y - ref).max()))
    for zb, yb in zip(z32.view(np.uint32).ravel().tolist(), y.view(np.uint32).ravel().tolist()):
        assert TANHF.setdefault(zb, yb) == yb, (tag, "tanhf of one z3 differs between routes", zb, yb, TANHF[zb])


# ------------------------------------------------------------------------------------------------------------ Part A data
def _pick(rng, vals, shape, p=None):
    return rng.choice(np.asarray(vals, np.float64), size=shape, p=p)


def exact_states(n, seed):
    """[9][n] float32 states on the 1/4 grid in [0, 1]; s[8] in {0, 1} flags the rows the saturation chain drives past |z3| = 13"""
    rng = np.random.default_rng(seed)
    s = np.zeros((9, n))
    s[:8] = _pick(rng, [0, 0.25, 0.5, 0.75, 1.0], (8, n), [0.3, 0.2, 0.2, 0.1, 0.2])
    s[8] = _pick(rng, [0.0, 1.0], n, [0.85, 0.15])
    return s.astype(np.float32)


@functools.lru_cache(maxsize=None)
def exact_actor(l1, l2, seed):
    """actor weights (Wt[in][out] float32) on which every act() route is exact on exact_states (module doc)"""
    rng = np.random.default_rng(7000 + seed)
    W1 = _pick(rng, [0, 0, 0, -1, -0.5, 0.5, 1], (9, l1))
    b1 = _pick(rng, [0, 0, -0.25, 0.25, 0.5], l1)
    W1[8] = 0.0
    u1, u2 = int(rng.integers(4, l1)), int(rng.integers(4, l2))
    W1[:, u1] = 0.0
    W1[8, u1] = 1.0
    b1[u1] = 0.0
    W1[:, :4] = 0.0                                   # z1 exactly 0 in every float4 lane
    b1[:4] = 0.0
    dens = min(1.0, 16.0 / l1)
    W2 = _pick(rng, [-0.25, -0.125, 0.125, 0.25], (l1, l2)) * (rng.uniform(size=(l1, l2)) < dens)
    b2 = _pick(rng, [0, 0, -0.125, -1 / 32, 1 / 32, 0.125], l2)
    W2[:, :4] = 0.0                                   # z2 exactly 0 in every float4 lane
    b2[:4] = 0.0
    W2[u1] = 0.0
    W2[:, u2] = 0.0
    W2[u1, u2] = 16.0
    b2[u2] = 0.0
    W3 = _pick(rng, [-2, -1, 1, 2], (l2, 2)) * (rng.uniform(size=(l2, 2)) < min(1.0, 24.0 / l2))
    W3[u2] = 0.0
    b3 = _pick(rng, [-0.25, -0.125, 0.125, 0.25], 2)
    # a power-of-two scale of W3 that spreads z3 over (-3, 3) off the flagged rows: root mean square in (1/2, 1]
    s = exact_states(512, 99).astype(np.float64)
    s[8] = 0
    h = np.maximum(np.maximum(s.T @ W1 + b1, 0) @ W2 + b2, 0)
    rms = float(np.sqrt(((h @ W3 + b3) ** 2).mean())) or 1.0
    W3 *= 2.0 ** np.floor(np.log2(1.0 / rms))
    W3[u2] = [1.0, -1.0]
    net = [(W1, b1), (W2, b2), (W3, b3)]
    return [(w.astype(np.float32), b.astype(np.float32)) for w, b in net]


ZERO, ONE = np.zeros(9, np.float32), np.ones(9, np.float32)


def exact_preconditions(actor, s):
    """the exactness conditions of Part A from the reference's intermediates; returns z3 [n][2] and the largest grid count"""
    net = f64(actor)
    (W1, b1), (W2, b2), (W3, b3) = net
    x = R.normalize(s, ZERO, ONE)
    np.testing.assert_array_equal(x, s.T.astype(np.float64))                    # normalisation is the identity
    f = R.forward(net, R.Val(x))
    assert tf32_exact(f["h1"].v) and tf32_exact(W2)                              # the TF32 layer-2 operands
    units = {"L1": grid_units(x, W1, b1), "L2": grid_units(f["h1"].v, W2, b2), "L3": grid_units(f["h2"].v, W3, b3)}
    for k, u in units.items():
        assert u < GRID_LIMIT, (k, u)
    for z in ("z1", "z2"):                                                       # relu(0) in every float4 lane
        zero = f[z].v == 0
        for lane in range(4):
            assert zero[:, lane::4].any(), (z, lane)
    z3 = f["z3"].v
    if s.shape[1] >= 64:
        assert (np.abs(z3) > 10).any() and (np.abs(z3) < 3).mean() > 0.5
        assert (z3 > 1).any() and (z3 < -1).any()
    assert np.array_equal(z3.astype(np.float32).astype(np.float64), z3)
    return z3, max(units.values())


# ------------------------------------------------------------------------------------------------------------ cases
SIMT_SMALL = {"ddpg_normalize_kernel", "gemm_batch_kernel<16,16>", "gemm_skinny_kernel"}
TF32_SMALL = {"ddpg_normalize_kernel", "gemm_batch_kernel<16,16>", "tc_gemm_kernel", "gemm_skinny_kernel"}
TF32_BIG = {"ddpg_normalize_kernel", "l1_fwd_kernel", "tc_gemm_kernel", "gemm_skinny_kernel"}
SIMT_BIG = {"ddpg_normalize_kernel", "l1_fwd_kernel", "gemm_batch_kernel<32,32>", "gemm_skinny_kernel"}
FUSED = {"ddpg_fused_act_kernel"}
EPI = {"ddpg_act_epilogue_kernel"}

# (id, route, n, l1, l2, use_tensor_cores, population, set_fused, forward kernels; the fused kernel has its epilogue inside)
CASES = [(f"fused_n{n}", "fused act cluster kernel", n, 250, 500, 0, 1, None, FUSED) for n in (1, 7, 8, 9, 63, 64)] + [
    ("fused_498", "fused act cluster kernel, W2 not vec16 (250/498)", 40, 250, 498, 0, 1, None, FUSED),
    ("simt_n65", "SIMT: gemm_batch<16,16> + gemm_skinny (n = 65 > 64, fused on)", 65, 250, 500, 0, 1, None, SIMT_SMALL),
    ("simt_unfused_n5", "SIMT with set_fused(False)", 5, 250, 500, 0, 1, False, SIMT_SMALL),
    ("simt_tc_n255", "SIMT on a TF32 handle, one row below TC_MIN_ROWS", 255, 250, 500, 1, 1, None, SIMT_SMALL),
    ("simt_big_n1024", "fp32 large: l1_fwd + gemm_batch<32,32> + gemm_skinny", 1024, 250, 500, 0, 1, None, SIMT_BIG),
    ("simt_24_20", "narrow net 24/20: output layer through gemm_batch", 200, 24, 20, 0, 1, False,
     {"ddpg_normalize_kernel", "gemm_batch_kernel<16,16>"}),
    ("tc_n256", "TF32: gemm_batch layer 1, tc_gemm layer 2", 256, 250, 500, 1, 1, None, TF32_SMALL),
    ("tc_n1000", "TF32, ragged last tile", 1000, 250, 500, 1, 1, None, TF32_SMALL),
    ("tc_n1024", "TF32 with l1_fwd", 1024, 250, 500, 1, 1, None, TF32_BIG),
    ("tc_100_132", "TF32 at 100/132: partial N tiles", 4096, 100, 132, 1, 1, None, TF32_BIG),
    ("tc_n131075", "TF32, 2^17 + 3 rows (a fixed subset compared)", 131075, 250, 500, 1, 1, None, TF32_BIG),
    ("tc_off_498", "use_tensor_cores = 1 with l2 % 4 != 0: SIMT", 4096, 250, 498, 1, 1, None, SIMT_BIG),
    ("pop_3x40", "population 3 x 40: SIMT", 40, 250, 500, 1, 3, None, SIMT_SMALL),
    ("pop_7x37", "population 7 x 37: TF32, 37-row tiles", 37, 250, 500, 1, 7, None, TF32_SMALL),
    ("pop_16x64", "population 16 x 64: TF32 + l1_fwd", 64, 250, 500, 1, 16, None, TF32_BIG),
    ("pop_80x100", "population 80 x 100: TF32 + l1_fwd", 100, 250, 500, 1, 80, None, TF32_BIG),
]
CASE_IDS = [c[0] for c in CASES]


def compared_rows(n):
    """every row, or for large n the first and last 512, the rows around every 128-row tile edge and every 257th row"""
    if n <= 8192:
        return np.arange(n)
    edges = np.arange(128, n, 128)
    rows = np.concatenate([np.arange(512), np.arange(n - 512, n), edges - 2, edges - 1, edges, edges + 1, np.arange(0, n, 257)])
    return np.unique(rows[(rows >= 0) & (rows < n)])


@pytest.mark.parametrize("l1,l2,n,seed", sorted({(c[3], c[4], min(c[2], 8192), s) for c in CASES for s in range(min(c[6], 3))}))
def test_exact_act_preconditions(l1, l2, n, seed):
    """the data Part A feeds every act() route is exact: TF32 operands, fp32 sums below 2^22 grid units, zeros in every lane,
    z3 spread over (-3, 3) with saturating rows (no GPU needed)"""
    z3, worst = exact_preconditions(exact_actor(l1, l2, seed), exact_states(max(n, 64), seed))
    print("%d/%d n=%d seed %d: largest sum |terms| / grid = 2^%.1f, |z3| > 10 on %d rows" % (l1, l2, n, seed, np.log2(max(worst, 1.0)),
                                                                                        int((np.abs(z3) > 10).any(1).sum())))


# ------------------------------------------------------------------------------------------------------------ device plumbing
@pytest.fixture
def learner_factory(monkeypatch):
    """Learner(...) with SHEMS_DDPG_FUSED unset for its creation, closed at the end of the test"""
    import shems_b200 as sb
    made = []

    def make(**kw):
        monkeypatch.delenv("SHEMS_DDPG_FUSED", raising=False)
        le = sb.Learner(params=sb.default_ddpg_params(**kw))
        made.append(le)
        return le

    yield make
    for le in made:
        le.close()


def make_case(learner_factory, case):
    name, route, n, l1, l2, tc, P, fused, kern = case
    le = learner_factory(l1=l1, l2=l2, use_tensor_cores=tc, population=P)
    if fused is not None:
        assert le.set_fused(fused) is fused
    return le


def to_soa(x):
    """[P][k][n] -> [k][P·n]"""
    P, k, n = x.shape
    return np.ascontiguousarray(x.transpose(1, 0, 2).reshape(k, P * n))


def from_soa(x, P):
    k, N = x.shape
    return np.ascontiguousarray(x.reshape(k, P, N // P).transpose(1, 0, 2))


def run_act(le, obs, P, soa, **kw):
    """le.act on obs [P][9][n] in the packed or the SoA layout -> (a, scaled) [P][2][n] (host)"""
    if P == 1:
        kw = {k: (dev(v[0]) if k == "noise" and v is not None else v) for k, v in kw.items()}
        a, s = le.act(dev(obs[0]), **kw)
        return host(a)[None], host(s)[None]
    if soa:
        kw = {k: (dev(to_soa(v)) if k == "noise" and v is not None else v) for k, v in kw.items()}
        a, s = le.act(dev(to_soa(obs)), soa=True, **kw)
        return from_soa(host(a), P), from_soa(host(s), P)
    kw = {k: (dev(v) if k == "noise" and v is not None else v) for k, v in kw.items()}
    a, s = le.act(dev(obs), **kw)
    return host(a), host(s)


def layouts(P):
    return (False, True) if P > 1 else (False,)


# ------------------------------------------------------------------------------------------------------------ Part A
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_act_route_bit_exact(learner_factory, case):
    """every learner gets its own exact weights; act(), act(soa) and act_ou (z = 0, X = 0) all return tanhf(z3) bit for bit"""
    name, route, n, l1, l2, tc, P, fused, kern = case
    le = make_case(learner_factory, case)
    rows = compared_rows(n)
    obs = np.stack([exact_states(n, 100 + l) for l in range(P)])
    z3 = []
    for l in range(P):
        actor = exact_actor(l1, l2, l)
        set_net(le.select(l), ACTOR, actor)
        le.set_norm(ZERO, ONE)
        z3.append(exact_preconditions(actor, obs[l][:, rows])[0])
    (a, _), got = kernels(lambda: run_act(le, obs, P, False, train=False))
    want = kern | (set() if kern == FUSED else EPI)
    print("\n%s: %s\n  kernels: %s" % (name, route, sorted(got)))
    assert got == want, (name, sorted(got), sorted(want))
    for l in range(P):
        record_tanhf(z3[l], a[l][:, rows].T, (name, l))
    for soa in layouts(P):
        a2, _ = run_act(le, obs, P, soa, noise=np.zeros((P, 2, n), np.float32))
        np.testing.assert_array_equal(a2, a, err_msg="%s caller noise 0, soa=%s" % (name, soa))
    ou_x = dev(np.zeros((P, 2, n) if P > 1 else (2, n), np.float32))
    z = dev(np.zeros((P, 2, n) if P > 1 else (2, n)))
    (a3, _), got = kernels(lambda: le.act_ou(dev(obs if P > 1 else obs[0]), ou_x, theta=0.15, mu=0.0, sigma=0.1, dt=1e-2, z=z))
    assert got == (kern - FUSED) | ({"ddpg_fused_act_kernel"} if kern == FUSED else set()) | {"ddpg_act_ou_epilogue_kernel"}, sorted(got)
    np.testing.assert_array_equal(host(a3).reshape(P, 2, n), a, err_msg="%s act_ou" % name)
    print("  every learner: tanhf(z3) bit-exact, within 2 ulp of tanh; act, act(noise = 0), act_ou agree%s" %
          (", packed and SoA" if P > 1 else ""))


@pytest.mark.gpu
def test_act_scratch_growth_bit_exact(learner_factory):
    """one TF32 handle acting on 1000, 70 000, 5, then 1000 states: the scratch grows, then serves smaller calls; every call checked"""
    le = learner_factory(use_tensor_cores=1)
    actor = exact_actor(250, 500, 0)
    set_net(le, ACTOR, actor)
    le.set_norm(ZERO, ONE)
    for k, n in enumerate((1000, 70000, 5, 1000)):
        s = exact_states(n, 300 + k)
        rows = compared_rows(n)
        z3, _ = exact_preconditions(actor, s[:, rows])
        a, _ = le.act(dev(s), train=False)
        record_tanhf(z3, host(a)[:, rows].T, ("scratch", n))


@pytest.mark.gpu
@pytest.mark.parametrize("via", ["rollout", "evaluate"])
def test_cluster_kernel_first_step_bit_exact(sb, train_series, via):
    """the first action of the persistent cluster kernel (actor_rollout.cu, -fmad=false) on exact start states is the tanhf(z3)
    every act() route gives"""
    n = 100
    le = sb.Learner()
    actor = exact_actor(250, 500, 0)
    set_net(le, ACTOR, actor)
    le.set_norm(ZERO, ONE)
    s = exact_states(n, 400)
    z3, _ = exact_preconditions(actor, s)
    env = sb.Shems(72, train_series, n_envs=n)
    env.reset(rng=1)
    env.set_state(s, env.idx)
    if via == "rollout":
        out, got = kernels(lambda: le.rollout(env, 1, want_actions=True))
    else:
        out, got = kernels(lambda: le.evaluate(env, 1, want_actions=True))
    assert got == {"actor_rollout_kernel"}, sorted(got)
    record_tanhf(z3, host(out["actions"][0]).T, via)


# ------------------------------------------------------------------------------------------------------------ Part B data
@pytest.fixture(scope="module")
def state_pool(sb, train_series):
    """(states [9][K] float32, s_min, s_max): random-policy rollouts of the train series and random_states corners; the norm from
    min_max_buffer over a sample of the rollouts, so some states lie outside it"""
    n, T = 512, 72
    env = sb.Shems(T, train_series, n_envs=n)
    mem = sb.Replay(n * T)
    env.reset(rng=3)
    out = env.rollout(sb.POLICY_RANDOM, T, seed=3, replay=mem, want_obs=True)
    obs = host(out["obs"]).transpose(1, 0, 2).reshape(9, -1)
    mn, mx = mem.min_max_buffer(2000, rng_mm=1)
    corners, _ = random_states(np.random.default_rng(5), 4096, train_series, sb._lib.params_for_charger(98))
    pool = np.concatenate([obs, corners], 1).astype(np.float32)
    lo, hi = pool.min(1), pool.max(1)
    assert np.any((lo < mn) | (hi > mx)), "some states lie outside [s_min, s_max]"
    return pool, mn, mx


def realistic_learner(le, l, rng, pool, z3_sd=2.5):
    """learner l: its init() actor with random biases and W3 scaled per output so that z3 spreads over the state pool with standard
    deviation z3_sd around a random centre (×40 on init() leaves the actions of these states in a narrow band), its own s_min / s_max
    (the pool's norm widened by up to half its span on either side, so that learners' norms differ widely) and its own noise_scale"""
    le.select(l)
    (W1, _), (W2, _), (W3, _) = get_net(le)
    l1, l2 = W2.shape
    b1, b2 = rng.normal(0, 0.05, l1).astype(np.float32), rng.normal(0, 0.05, l2).astype(np.float32)
    states, mn, mx = pool
    span = mx - mn
    lo = (mn - span * rng.uniform(0, 0.5, 9)).astype(np.float32)
    hi = (mx + span * rng.uniform(0, 0.5, 9)).astype(np.float32)
    sample = states[:, rng.integers(0, states.shape[1], 2048)]
    z = R.forward(f64([(W1, b1), (W2, b2), (W3, np.zeros(2, np.float32))]), R.Val(R.normalize(sample, lo, hi)))["z3"].v
    c = z3_sd / z.std(0)
    W3 = (W3 * c[None, :]).astype(np.float32)
    b3 = (-c * z.mean(0) + rng.normal(0, 0.5, 2)).astype(np.float32)
    actor = [(W1, b1), (W2, b2), (W3, b3)]
    set_net(le, ACTOR, actor)
    le.set_norm(lo, hi)
    le.set_hparams(noise_scale=float(rng.uniform(0.5, 2.0)))
    return dict(actor=f64(actor), lo=lo, hi=hi, ns=np.float32(le.get_hparams()["noise_scale"]))


def draw_states(pool, n, rng):
    return pool[0][:, rng.integers(0, pool[0].shape[1], n)]


# ------------------------------------------------------------------------------------------------------------ Part B
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_act_route_within_bound(learner_factory, state_pool, case):
    """realistic weights, states and norms; Philox noise with per-learner noise_scale and env_id_base != 0: every action element of
    every learner, packed and SoA, within C_BOUND × its bound"""
    name, route, n, l1, l2, tc, P, fused, kern = case
    le = make_case(learner_factory, case)
    le.init(11)
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    ls = [realistic_learner(le, l, rng, state_pool) for l in range(P)]
    obs = np.stack([draw_states(state_pool, n, rng) for _ in range(P)])
    rows = compared_rows(n)
    seed, step, sigma = 4242, 3, 0.1
    worst = 0.0
    for soa in layouts(P):
        (a, _), got = kernels(lambda: run_act(le, obs, P, soa, train=True, sigma=sigma, rng_act=seed, step=step, env_id_base=E_BASE))
        assert got == kern | (set() if kern == FUSED else EPI), sorted(got)
        for l in range(P):
            y = R.actor_out(ls[l]["actor"], ls[l]["lo"], ls[l]["hi"], obs[l][:, rows], track=True, tf32="tc_gemm_kernel" in kern)
            nz = gauss_noise(seed, E_BASE + l * n + rows, step, sigma_eff(sigma, ls[l]["ns"])).T
            worst = max(worst, check_bounded(a[l][:, rows].T, y, nz, (name, l, soa)))
    print("\n%s: %s\n  kernels: %s\n  largest err / bound: %.3f, |a| = 1 on %.1f%% of the actions" %
          (name, route, sorted(got), worst, 100 * (np.abs(a) == 1).mean()))


# ------------------------------------------------------------------------------------------------------------ epilogues
EPI_ROUTES = [("fused", 40, 0, 1, FUSED), ("simt", 100, 0, 1, SIMT_SMALL | EPI), ("tc_pop", 64, 1, 4, TF32_SMALL | EPI)]


@pytest.mark.gpu
@pytest.mark.parametrize("route", EPI_ROUTES, ids=[r[0] for r in EPI_ROUTES])
def test_act_epilogues_bit_exact(learner_factory, state_pool, route):
    """given the route's own y (caller noise 0): caller noise, scale_action with non-default bounds, the OU step and the Philox
    Box–Muller noise, restated in numpy"""
    name, n, tc, P, kern = route
    lo, hi = (-0.75, 0.125), (2.5, 0.875)
    le = learner_factory(use_tensor_cores=tc, population=P, act_lo=lo, act_hi=hi)
    le.init(12)
    rng = np.random.default_rng(len(name))
    ls = [realistic_learner(le, l, rng, state_pool) for l in range(P)]
    obs = np.stack([draw_states(state_pool, n, rng) for _ in range(P)])
    (y, _), got = kernels(lambda: run_act(le, obs, P, False, noise=np.zeros((P, 2, n), np.float32)))
    assert got == kern, sorted(got)
    assert np.abs(y).max() <= 1 and (np.abs(y) >= 0.5).any() and (np.abs(y) < 0.5).any()
    lo32, hi32 = np.float32(lo), np.float32(hi)
    sc = lambda a: np.stack([scale_action(a[..., k, :], lo32[k], hi32[k]) for k in range(2)], -2)
    for soa in layouts(P):
        # caller noise: past ±1, exactly onto ±1 (1 - y is exact for |y| >= 1/2), small values
        nz = rng.normal(0, 0.3, y.shape).astype(np.float32)
        big = np.abs(y) >= 0.5
        onto = big & (rng.uniform(size=y.shape) < 0.3)
        nz = np.where(onto, np.sign(y) - y, nz)
        nz = np.where(big & ~onto & (rng.uniform(size=y.shape) < 0.3), 2 * np.sign(y), nz).astype(np.float32)
        assert ((y + nz) == np.sign(y)).any() and (np.abs(y + nz) > 1).any()
        a, s = run_act(le, obs, P, soa, noise=nz)
        want = np.clip(y + nz, np.float32(-1), np.float32(1))
        np.testing.assert_array_equal(a, want, err_msg="%s caller noise soa=%s" % (name, soa))
        np.testing.assert_array_equal(s, sc(want), err_msg="%s scaled soa=%s" % (name, soa))
        # Philox: within one ulp of the numpy Box–Muller noise, σ_eff = RN32(σ · noise_scale_l)
        seed, step, sigma = 99, 5, 0.3
        a, s = run_act(le, obs, P, soa, train=True, sigma=sigma, rng_act=seed, step=step, env_id_base=E_BASE)
        for l in range(P):
            nzl = gauss_noise(seed, E_BASE + l * n + np.arange(n), step, sigma_eff(sigma, ls[l]["ns"]))
            a_lo, a_hi = noisy_interval(y[l], nzl)
            assert np.all((a[l] >= a_lo) & (a[l] <= a_hi)), (name, l, soa)
            np.testing.assert_array_equal(s[l], sc(a[l]))
        # no noise: σ = 0, and noise_scale = 0 with σ > 0
        a, _ = run_act(le, obs, P, soa, train=True, sigma=0.0, rng_act=seed, step=step, env_id_base=E_BASE)
        np.testing.assert_array_equal(a, y)
        for l in range(P):
            le.select(l).set_hparams(noise_scale=0.0)
        a, _ = run_act(le, obs, P, soa, train=True, sigma=sigma, rng_act=seed, step=step, env_id_base=E_BASE)
        np.testing.assert_array_equal(a, y)
        for l in range(P):
            le.select(l).set_hparams(noise_scale=float(ls[l]["ns"]))
    # OU with caller z over several steps: dx = θ(μ - X)dt in Float32, + Float32(σ√dt)·z in Float64, X += dx
    theta, mu, sigma, dt = np.float32(0.15), np.float32(0.05), np.float32(0.2), np.float32(1e-2)
    X = rng.normal(0, 0.5, y.shape).astype(np.float32)
    ou = dev(X if P > 1 else X[0])
    for t in range(4):
        z = rng.normal(0, 1, y.shape) * (4 if t == 3 else 1)
        a, s = le.act_ou(dev(obs if P > 1 else obs[0]), ou, theta=float(theta), mu=float(mu), sigma=float(sigma), dt=float(dt),
                         z=dev(z if P > 1 else z[0]))
        a, s = host(a).reshape(y.shape), host(s).reshape(y.shape)
        for l in range(P):
            ssd = np.float32(sigma_eff(sigma, ls[l]["ns"]) * np.sqrt(dt))
            dx = np.float32(np.float32(theta * np.float32(mu - X[l])) * dt)
            dx = (dx.astype(np.float64) + np.float64(ssd) * z[l]).astype(np.float32)
            X[l] = X[l] + dx
        np.testing.assert_array_equal(host(ou).reshape(y.shape), X, err_msg="%s OU X step %d" % (name, t))
        want = np.clip(y + X, np.float32(-1), np.float32(1))
        np.testing.assert_array_equal(a, want, err_msg="%s OU a step %d" % (name, t))
        np.testing.assert_array_equal(s, sc(want), err_msg="%s OU scaled step %d" % (name, t))
    print("\n%s: kernels %s; caller noise, scaled, Philox (1 ulp) and 4 OU steps exact" % (name, sorted(got)))


# ------------------------------------------------------------------------------------------------------------ evaluation, inference, episodes
def follow(sb, series, start, idx, n_steps, actions, check, env_kw=None):
    """replay a run from (start, idx) through Shems.step with the kernel's own actions (scale_action with the default bounds 0 / 1);
    check(t, s) on every step's state; returns the final state"""
    env = sb.Shems(n_steps, series, n_envs=start.shape[1], **(env_kw or {}))
    env.set_state(start, idx)
    for t in range(n_steps):
        s = env.state
        check(t, s)
        env.step(dev(scale_action(actions[t], 0.0, 1.0)))
    return env.state


def actor_ref(le, l, net=ACTOR):
    le.select(l)
    st, _ = le.get_state()
    return f64(get_net(le, net)), st[-18:-9].copy(), st[-9:].copy()


def negate_w3(le, l):
    """learner l's actor with the output layer's weights negated: another actor, its outputs as spread"""
    le.select(l)
    layers = get_net(le)
    layers[2] = (-layers[2][0], layers[2][1])
    set_net(le, ACTOR, layers)


@pytest.mark.gpu
@pytest.mark.parametrize("n,sigma", [(1, 0.0), (13, 0.0), (100, 0.0), (1, 0.1), (13, 0.1), (100, 0.1), (1, None)],
                         ids=["n1", "n13", "n100", "n1_noise", "n13_noise", "n100_noise", "inference_test_set"])
def test_rollout_cluster_kernel_open_loop(sb, train_series, charger98_test_series, state_pool, n, sigma):
    """ddpg_rollout on one learner (the persistent cluster kernel): every step's action against actor_out on that step's state
    (+ the re-derived noise), the run replayed through Shems.step bit for bit.  inference_test_set: reset!(rng = -1) and the whole
    test series (nrows - 1 steps)"""
    le = sb.Learner()
    le.init(21)
    rng = np.random.default_rng(n)
    ns = realistic_learner(le, 0, rng, state_pool)["ns"]
    inference = sigma is None
    ser = charger98_test_series if inference else train_series
    T = ser.shape[1] - 1 if inference else 72
    env = sb.Shems(T, ser, n_envs=n, env_id_base=E_BASE)
    env.reset(rng=-1 if inference else 7)
    s0, i0 = env.state, env.idx
    seed = 31
    out, got = kernels(lambda: le.rollout(env, T, sigma=sigma or 0.0, rng_ep=seed, want_actions=True))
    assert got == {"actor_rollout_kernel"}, sorted(got)
    acts = host(out["actions"])
    actor, lo, hi = actor_ref(le, 0)
    se = sigma_eff(sigma or 0.0, ns)
    worst = [0.0]

    def check(t, s):
        y = R.actor_out(actor, lo, hi, s, track=True, tf32=False)
        nz = gauss_noise(rng_step(seed, t + 1), E_BASE + np.arange(n), t + 1, se).T if sigma else None
        worst[0] = max(worst[0], check_bounded(acts[t].T, y, nz, ("rollout", n, sigma, t)))

    end = follow(sb, ser, s0, i0, T, acts, check, dict(env_id_base=E_BASE))
    np.testing.assert_array_equal(end, env.state)
    print("\nrollout n=%d sigma=%s T=%d: kernels %s, largest err / bound %.3f, |a| = 1 on %.1f%% of the actions" %
          (n, sigma, T, sorted(got), worst[0], 100 * (np.abs(acts) == 1).mean()))


@pytest.mark.gpu
def test_evaluate_population_open_loop(sb, train_series, state_pool):
    """ddpg_evaluate on P = 5 learners × 13 instances (ragged 8-instance clusters), each with its own norm and weights, for ACTOR and
    for ACTOR_BEST after keep_best (the actors are changed afterwards, so the two differ)"""
    import torch
    P, n, T = 5, 13, 72
    pop = sb.Learner(params=sb.default_ddpg_params(population=P))
    pop.init(5)
    rng = np.random.default_rng(55)
    for l in range(P):
        realistic_learner(pop, l, rng, state_pool)
    env = sb.Shems(T, train_series, n_envs=P * n, env_id_base=E_BASE)
    env.reset(rng=17)
    s0, i0 = env.state, env.idx
    pop.keep_best(torch.full((P * n,), 1e30, dtype=torch.float64, device="cuda"), n, 1)
    best = [actor_ref(pop, l, ACTOR_BEST) for l in range(P)]
    for l in range(P):
        negate_w3(pop, l)
    cur = [actor_ref(pop, l) for l in range(P)]
    for b, refs in ((False, cur), (True, best)):
        env.set_state(s0, i0)
        out, got = kernels(lambda: pop.evaluate(env, T, best=b, want_actions=True))
        assert got == {"actor_rollout_kernel"}, sorted(got)
        acts = host(out["actions"])
        worst = [0.0]

        def check(t, s):
            for l, (actor, _, _) in enumerate(refs):
                lo, hi = cur[l][1], cur[l][2]
                sl = slice(l * n, (l + 1) * n)
                y = R.actor_out(actor, lo, hi, s[:, sl], track=True, tf32=False)
                worst[0] = max(worst[0], check_bounded(acts[t][:, sl].T, y, None, ("evaluate", b, l, t)))

        end = follow(sb, train_series, s0, i0, T, acts, check)
        np.testing.assert_array_equal(end, env.state)
        print("\nevaluate P=%d x %d best=%s: largest err / bound %.3f" % (P, n, b, worst[0]))
    assert not np.array_equal(best[0][0][2][0], cur[0][0][2][0])


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["pop_3x100_tf32", "wide_64_640"])
def test_rollout_fallback_open_loop(sb, train_series, state_pool, shape):
    """ddpg_rollout where the cluster kernel does not apply: one act + step! launch pair per step (a TF32 population; a net wider
    than the cluster kernel's plan), with Philox noise keyed by env_id_base + l·n + j"""
    if shape == "pop_3x100_tf32":
        P, n, kw, kern = 3, 100, dict(population=3, use_tensor_cores=1), TF32_SMALL | EPI
    else:
        P, n, kw, kern = 1, 9, dict(l1=64, l2=640, batch=32), SIMT_SMALL | EPI
    le = sb.Learner(params=sb.default_ddpg_params(**kw))
    le.init(2)
    rng = np.random.default_rng(P)
    ls = [realistic_learner(le, l, rng, state_pool) for l in range(P)]
    T, seed, sigma = 24, 8, 0.1
    env = sb.Shems(72, train_series, n_envs=P * n, env_id_base=E_BASE)
    env.reset(rng=4)
    s0, i0 = env.state, env.idx
    out, got = kernels(lambda: le.rollout(env, T, sigma=sigma, rng_ep=seed, want_actions=True))
    assert kern <= got and "actor_rollout_kernel" not in got, sorted(got)
    acts = host(out["actions"])
    worst = [0.0]

    def check(t, s):
        for l in range(P):
            sl = slice(l * n, (l + 1) * n)
            y = R.actor_out(ls[l]["actor"], ls[l]["lo"], ls[l]["hi"], s[:, sl], track=True, tf32="tc_gemm_kernel" in kern)
            nz = gauss_noise(rng_step(seed, t + 1), E_BASE + l * n + np.arange(n), t + 1, sigma_eff(sigma, ls[l]["ns"])).T
            worst[0] = max(worst[0], check_bounded(acts[t][:, sl].T, y, nz, (shape, l, t)))

    end = follow(sb, train_series, s0, i0, T, acts, check, dict(env_id_base=E_BASE))
    np.testing.assert_array_equal(end, env.state)
    print("\n%s: kernels %s, largest err / bound %.3f" % (shape, sorted(got), worst[0]))


EPISODES = [("fused_n8_gn", 1, 8, 0, "gn"), ("tc_pop_4x64_gn", 4, 64, 1, "gn"), ("fused_n8_ou", 1, 8, 0, "ou")]


@pytest.mark.gpu
@pytest.mark.parametrize("case", EPISODES, ids=[c[0] for c in EPISODES])
def test_episode_acts_open_loop(sb, train_series, state_pool, case):
    """ddpg_episode with lr_actor = 0 (the critic still trains): the actor is bit-identical afterwards, and every ring transition's
    a is the reference on its s plus the re-derived noise.  ou: X is followed per instance, with a bound for the numpy Box–Muller"""
    from shems_b200.ddpg import push_groups
    name, P, n, tc, kind = case
    le = sb.Learner(params=sb.default_ddpg_params(population=P, use_tensor_cores=tc))
    le.init(3)
    rng = np.random.default_rng(P * n)
    ls = [realistic_learner(le, l, rng, state_pool) for l in range(P)]
    for l in range(P):
        le.select(l).set_hparams(lr_actor=0.0)
    theta, mu, dt = 0.15, 0.0, 1e-2
    if kind == "ou":
        le.set_noise("ou", theta=theta, mu=mu, dt=dt)
    T, seed, sigma, pre = 16, 6, 0.2, 256
    mems = [sb.Replay(pre + n * T) for _ in range(P)]
    s_pre = draw_states(state_pool, P * pre, rng)
    push_groups(mems, dev(s_pre), dev(rng.uniform(-1, 1, (2, P * pre)).astype(np.float32)), dev(rng.uniform(-3, 0, P * pre).astype(np.float32)),
                dev(draw_states(state_pool, P * pre, rng)))
    before = [get_net(le.select(l)) for l in range(P)]
    env = sb.Shems(72, train_series, n_envs=P * n, env_id_base=E_BASE)
    env.reset(rng=9)
    _, got = kernels(lambda: le.episode(env, mems if P > 1 else mems[0], T, train=True, sigma=sigma, rng_ep=seed, updates_per_step=1))
    act_kern = (FUSED if P == 1 else TF32_SMALL | EPI) | ({"ddpg_act_ou_epilogue_kernel"} if kind == "ou" else set())
    assert act_kern <= got and (kind == "ou") == ("ddpg_act_ou_epilogue_kernel" in got), sorted(got)
    worst = 0.0
    for l in range(P):
        for (w0, b0), (w1, b1) in zip(before[l], get_net(le.select(l))):
            np.testing.assert_array_equal(w0, w1)
            np.testing.assert_array_equal(b0, b1)
        s, a, _, _, _ = mems[l].get()
        s, a = s[:, pre:].reshape(9, T, n), a[:, pre:].reshape(2, T, n)
        X, eX = np.zeros((2, n), np.float32), np.zeros((2, n))
        se = sigma_eff(sigma, ls[l]["ns"])
        for t in range(T):
            ids = E_BASE + l * n + np.arange(n)
            y = R.actor_out(ls[l]["actor"], ls[l]["lo"], ls[l]["hi"], s[:, t], track=True, tf32="tc_gemm_kernel" in act_kern)
            if kind == "gn":
                nz = gauss_noise(rng_step(seed, t + 1), ids, t + 1, se)
                worst = max(worst, check_bounded(a[:, t].T, y, nz.T, (name, l, t)))
                continue
            z = standard_normals(rng_step(seed, t + 1), ids, t + 1)
            ssd = np.float32(se * np.sqrt(np.float32(dt)))
            dx = np.float32(np.float32(np.float32(theta) * np.float32(np.float32(mu) - X)) * np.float32(dt))
            dx = (dx.astype(np.float64) + np.float64(ssd) * z).astype(np.float32)
            X = X + dx
            # a z that differs in its last bits may flip the two roundings: carry that as a bound on X
            eX = eX * (1 + theta * dt) + 2 * (np.spacing(np.abs(dx)) + np.spacing(np.abs(X)))
            ys = y.v.T + X
            bound = y.err.T + eX + R.U_FP32 * np.abs(ys)
            err = np.abs(a[:, t].astype(np.float64) - np.clip(ys, -1, 1))
            assert np.all(err <= C_BOUND * bound), (name, l, t, float((err / bound).max()))
            worst = max(worst, float((err / (C_BOUND * bound)).max()))
        if kind == "ou":
            xs = le.get_ou_state()
            assert np.all(np.abs(xs[:, l * n:(l + 1) * n] - X) <= eX), (name, l)
    print("\n%s: act kernels %s; actor unchanged, every transition's action within the bound (largest err / bound %.3f)" %
          (name, sorted(act_kern), worst))
