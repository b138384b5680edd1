"""Sampling-fraction learning record by record: the replay of the renderer (adam_hist -> exclusive_scan -> adam_scatter -> adam_seq -> adam_progress, and
adam_pack / adam_merge across replicas, csrc/ppg_kernels.cuh) against the reference's AdamOptimizer (GP:69-133) driven through
optimizeBsdfSamplingFraction (GP:672-697) on the same records in the same order.

Every float comparison has three sides: the replay under test (the CUDA kernels with -m gpu; the same device source compiled for the host otherwise),
the reference in float32 (the reference's own code from oracle/_ref where it was built, else the oracle's restatement, bit-equal to it:
tests/test_oracle_sdtree.py), and the reference's formulas evaluated in float64 here as the arbiter.  The float64 replay accumulates the batch
weight in float32 like both others, so all three take their Adam steps at the same records and `iter` / `batchAcc` must agree exactly; m, v, theta and
batchGrad must satisfy |dut - ref64| <= 4 |ref32 - ref64| + floor, i.e. the replay may be as far from exact arithmetic as the reference itself
(times 4), plus a floor for the roundings the two float32 sides take at different places.

Record domain (where the reference itself stays finite): pdfs in [1e-4, 1e8], product in [1e-3, 1], weights in (0, 1], theta in [-20, 20]."""
import ctypes as C
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle_lib as O
from common import ROOT

f32p = C.POINTER(C.c_float)
CUDA_INC = next((p for p in (os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include"), "/usr/local/cuda/include") if os.path.exists(os.path.join(p, "cuda_runtime.h"))), None)
LOSSES = ["kl", "var"]
LOSS_CODE = {"kl": 1, "var": 2}
B1, B2, EPS, LR = float(np.float32(0.9)), float(np.float32(0.999)), float(np.float32(1e-8)), float(np.float32(0.01))   # the reference's float hyperparameters

# Floors of |dut - ref64| beyond 4 |ref32 - ref64|, per field: theta absolute; m, batchGrad relative to the leaf's gradient scale sqrt(v) + |m|;
# v relative to v.  Measured spread (largest excess over 4 |ref32 - ref64| across all cases below, both losses):
#   host-compiled replay (exact division, host expf):  theta 1.0e-7, m 2.3e-5, v 1.2e-5, batchGrad 1.6e-5
#   B200 (sm_100a, __fdividef / __expf), three runs:    theta <= 5.7e-7, m <= 3.4e-4, v <= 6.9e-5, batchGrad <= 1.5e-4
# The device's spread on m / v / batchGrad changes from run to run with the bucket order the scatter's atomics produce (the reference is replayed
# in that order), hence floors of about 3x the largest seen; theta, the quantity that steers sampling, stays below 1e-6.
FLOOR = {"theta": 1e-4, "m": 1e-3, "v": 3e-4, "batchGrad": 1e-3}


# ------------------------------------------------------------------------------------------------------------------- cases
START = {   # iter, m, v, variable, batchAcc, batchGrad
    "fresh": (0, 0, 0, 0, 0, 0),
    "theta +20": (40, 0.05, 0.01, 20.0, 0, 0), "theta -20": (40, -0.05, 0.01, -20.0, 0, 0),
    "theta +17": (40, 0.05, 0.01, 17.0, 0, 0), "theta -17": (40, -0.05, 0.01, -17.0, 0, 0),
    "theta +16.5": (40, 0.05, 0.01, 16.5, 0, 0), "theta -16.5": (40, -0.05, 0.01, -16.5, 0, 0),
    "iter 1e6": (1e6, 0.3, 2.0, 1.5, 0, 0),
    "carried batch": (12, -0.2, 0.5, -0.7, 0.75, -0.4),
}
SIZES = [0, 1, 31, 32, 33, 64, 65]                 # records per leaf: the 32-record prefetch chunk edges
WEIGHTS = ["one", "half", "box", "mix"]            # 1.0 | 0.5 (kickstart NEE: 0.5 + 0.5 is not > 1) | box-filter fractions in (0, 1] | a mix
PDFS = ["loguniform", "equal", "dtree zero", "dtree over 2^25 bsdf"]


def _logu(rng, lo, hi, n):
    return np.exp(rng.uniform(math.log(lo), math.log(hi), n)).astype(np.float32)


def _records(rng, leaf, n, weights, pdfs):
    """n records of S-tree node `leaf` as record_into_leaf appends them: rec_a {bits(leaf), product, woPdf, bsdfPdf}, rec_b {dTreePdf, weight}."""
    a = np.zeros((n, 4), np.float32); b = np.zeros((n, 2), np.float32)
    a[:, 0] = np.full(n, leaf, np.uint32).view(np.float32)
    a[:, 1] = _logu(rng, 1e-3, 1.0, n); a[:, 2] = _logu(rng, 1e-4, 1e8, n); a[:, 3] = _logu(rng, 1e-4, 1e8, n)
    b[:, 0] = _logu(rng, 1e-4, 1e8, n)
    kind = np.full(n, PDFS.index(pdfs)) if pdfs != "mixed" else rng.integers(0, len(PDFS), n)
    eq = kind == 1; b[eq, 0] = a[eq, 3]
    b[kind == 2, 0] = 0.0
    big = kind == 3; a[big, 3] = _logu(rng, 1e-4, 1.0, int(big.sum())); b[big, 0] = a[big, 3] * np.float32(2.0 ** 25) * _logu(rng, 1.0, 1e3, int(big.sum()))
    w = {"one": np.ones(n), "half": np.full(n, 0.5), "box": rng.uniform(0, 1, n)}
    w["box"] = np.maximum(w["box"], 1e-3)
    wk = rng.integers(0, 3, n) if weights == "mix" else np.full(n, ["one", "half", "box"].index(weights))
    b[:, 1] = np.choose(wk, [w["one"], w["half"], w["box"]]).astype(np.float32)
    return a, b


def make_case(name, seed=1):
    """(states (L, 6), rec_a (n, 4), rec_b (n, 2)).  'grid': every start state x bucket size x weight kind x pdf kind (1008 leaves, records of all leaves
    interleaved); 'hot': one leaf with 2 10^5 records, stored contiguously (every warp of the bucketing kernels sees one leaf), next to a few small ones;
    'many': 70 000 leaves (past 16-bit indices and the scan's 1024-entry chunks) of 0..3 records; 'saturated': theta = +20 / +17 leaves fed only records
    with dTreePdf > 2^25 bsdfPdf."""
    rng = np.random.default_rng(seed)
    starts, A, Bb = [], [], []
    if name == "grid":
        for s in START.values():
            for n in SIZES:
                for w in WEIGHTS:
                    for p in PDFS:
                        a, b = _records(rng, len(starts), n, w, p); starts.append(s); A.append(a); Bb.append(b)
        a, b = np.concatenate(A), np.concatenate(Bb); perm = rng.permutation(len(a)); a, b = a[perm], b[perm]
    elif name == "hot":
        for k, s in enumerate(list(START.values())[:4]):
            a, b = _records(rng, k, 200000 if k == 0 else 40, "mix", "mixed"); starts.append(s); A.append(a); Bb.append(b)
        a, b = np.concatenate(A), np.concatenate(Bb)
    elif name == "many":
        L = 70000
        starts = [list(START.values())[i % len(START)] for i in range(L)]
        cnt = rng.integers(0, 4, L); leaf = np.repeat(np.arange(L), cnt); n = len(leaf)
        a, b = _records(rng, 0, n, "mix", "mixed"); a[:, 0] = leaf.astype(np.uint32).view(np.float32)
        perm = rng.permutation(n); a, b = a[perm], b[perm]
    elif name == "saturated":
        for k, (s, w) in enumerate([(START["theta +20"], "one"), (START["theta +20"], "half"), (START["theta +17"], "box"), (START["theta +17"], "one")]):
            a, b = _records(rng, k, 400, w, "dtree over 2^25 bsdf"); starts.append(s); A.append(a); Bb.append(b)
        a, b = np.concatenate(A), np.concatenate(Bb)
    else:
        raise ValueError(name)
    return np.asarray(starts, np.float32), np.ascontiguousarray(a), np.ascontiguousarray(b)


def leaf_of(a):
    return np.ascontiguousarray(a[:, 0]).view(np.uint32)


# ------------------------------------------------------------------------------------------------------------------- the two references
def _truth_kind():
    """The reference's own code (oracle/_ref) where it was built with ppgo_tree_set_adam; the oracle's restatement, bit-equal to it, otherwise."""
    return "ref" if O.have_ref() and hasattr(O.load("ref"), "ppgo_tree_set_adam") else "port"


def ref32_replay(states, a, b, loss):
    """The reference in float32: each leaf's records in the given order through DTreeWrapper::record (is_delta, so only optimizeBsdfSamplingFraction
    runs) on a one-leaf S-tree seeded with the leaf's state -- the leaves are independent, so one tree serves them all in turn."""
    o = O.Oracle(O.default_params(), aabb=((0, 0, 0), (1, 1, 1)), kind=_truth_kind())
    lib, h = o.lib, o.h
    out = np.array(states, np.float32, copy=True)
    leaf = leaf_of(a); order = np.argsort(leaf, kind="stable"); ls = leaf[order]
    cols = [np.ascontiguousarray(x, np.float32) for x in (a[order, 1], a[order, 2], a[order, 3], b[order, 0], b[order, 1])]
    n = len(order)
    pos = np.full((max(n, 1), 3), 0.5, np.float32); d = np.tile(np.float32([0, 0, 1]), (max(n, 1), 1)); rad = np.zeros(max(n, 1), np.float32)
    delta = np.ones(max(n, 1), np.uint8); st = np.zeros(6, np.float32)
    at = lambda arr, i, k=1: C.cast(int(arr.ctypes.data + arr.itemsize * k * int(i)), f32p)
    starts = np.flatnonzero(np.r_[True, ls[1:] != ls[:-1]]) if n else []
    for i0, i1 in zip(starts, list(starts[1:]) + [n]):
        l = int(ls[i0])
        o.set_adam(0, out[l])
        lib.ppgo_tree_record(h, int(i1 - i0), at(pos, i0, 3), at(d, i0, 3), at(rad, i0), at(cols[0], i0), at(cols[1], i0), at(cols[2], i0), at(cols[3], i0),
                             at(cols[4], i0), C.cast(int(delta.ctypes.data + int(i0)), C.POINTER(C.c_uint8)), None, 0, 0, LOSS_CODE[loss])
        lib.ppgo_tree_export(h, 0, None, None, None, None, None, None, None, None, None, None, st.ctypes.data_as(f32p), None)
        out[l] = st
    o.close()
    return out


def _f32(x):
    return float(np.float32(x))


def ref64_replay(states, a, b, loss):
    """GP:85-109 / 672-697 in float64 (the arbiter), hyperparameters at their float values; the batch weight is accumulated in float32 (a float add of
    float weights: computed in double and rounded once, which is exact float addition), so the steps fall on the same records as on the float32 sides."""
    p = 1.0 if loss == "kl" else 2.0
    out = np.array(states, np.float64, copy=True)
    leaf = leaf_of(a); order = np.argsort(leaf, kind="stable")
    prod, wo, bs = (a[order, k].astype(np.float64).tolist() for k in (1, 2, 3))
    dt, w = (b[order, k].astype(np.float64).tolist() for k in (0, 1))
    ls = leaf[order].tolist()
    i, n = 0, len(ls)
    while i < n:
        l = ls[i]
        it, m1, m2, th, acc, bg = out[l].tolist(); it = int(it)
        while i < n and ls[i] == l:
            f = 1.0 / (1.0 + math.exp(-th))
            mix = f * bs[i] + (1.0 - f) * dt[i]
            dl = -((prod[i] / mix) ** p) / wo[i] * (bs[i] - dt[i])
            g = dl * (f * (1.0 - f)) + 0.01 * th
            bg += g * w[i]; acc = _f32(acc + w[i])
            if acc > 1.0:
                grad = bg / acc
                it += 1
                lr = LR * math.sqrt(1.0 - B2 ** it) / (1.0 - B1 ** it)
                m1 = B1 * m1 + (1.0 - B1) * grad
                m2 = B2 * m2 + (1.0 - B2) * grad * grad
                th = min(max(th - lr * m1 / (math.sqrt(m2) + EPS), -20.0), 20.0)
                bg = 0.0; acc = 0.0
            i += 1
        out[l] = (it, m1, m2, th, acc, bg)
    return out


def spread(dut, r32, r64):
    """Largest excess of |dut - ref64| over 4 |ref32 - ref64| per field, in the units of FLOOR."""
    dut = dut.astype(np.float64); r32 = r32.astype(np.float64)
    scale = np.sqrt(np.abs(r64[:, 2])) + np.abs(r64[:, 1])
    ex = lambda c: np.abs(dut[:, c] - r64[:, c]) - 4 * np.abs(r32[:, c] - r64[:, c])
    with np.errstate(divide="ignore", invalid="ignore"):
        rel = lambda x, s: np.where(x > 0, x / np.where(s > 0, s, np.inf), 0.0)
        return {"theta": float(max(ex(3).max(initial=0), 0)), "m": float(rel(ex(1), scale).max(initial=0)),
                "v": float(rel(ex(2), np.abs(r64[:, 2])).max(initial=0)), "batchGrad": float(rel(ex(5), scale + np.abs(r64[:, 5])).max(initial=0))}


def assert_states(dut, r32, r64, what=""):
    print("spread", what, spread(dut, r32, r64))
    assert np.isfinite(dut).all() and np.isfinite(r32).all() and np.isfinite(r64).all(), what
    assert np.array_equal(dut[:, 0], r32[:, 0]) and np.array_equal(dut[:, 4], r32[:, 4]), what          # iter, batchAcc: exact
    assert np.array_equal(r64[:, 0], r32[:, 0]) and np.array_equal(r64[:, 4], r32[:, 4].astype(np.float64)), what
    s = spread(dut, r32, r64)
    bad = {k: v for k, v in s.items() if v > FLOOR[k]}
    assert not bad, (what, s)
    return s


# ------------------------------------------------------------------------------------------------------------------- host-compiled replay (CPU)
@pytest.fixture(scope="module")
def hostdev(tmp_path_factory):
    if CUDA_INC is None or shutil.which("g++") is None:
        pytest.skip("needs g++ and the CUDA headers")
    so = str(tmp_path_factory.mktemp("hostdev") / "libdevice_on_host.so")
    cmd = ["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I" + CUDA_INC, "-D__device__=", "-D__host__=", "-D__global__=", "-D__shared__=",
           "-D__forceinline__=inline", "-D__noinline__=", "-D__launch_bounds__(...)=", "-Wno-unused-function", os.path.join(ROOT, "tests", "hostdev", "device_on_host.cpp"), "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    lib = C.CDLL(so)
    lib.dev_fraction_replay.argtypes = [f32p, C.c_size_t, f32p, f32p, C.c_size_t, C.c_int]
    return lib


def host_replay(lib, states, a, b, loss):
    st = np.array(states, np.float32, copy=True)
    assert lib.dev_fraction_replay(st.ctypes.data_as(f32p), len(st), a.ctypes.data_as(f32p), b.ctypes.data_as(f32p), len(a), LOSS_CODE[loss]) == 0
    return st


@pytest.mark.parametrize("loss", LOSSES)
@pytest.mark.parametrize("case", ["grid", "hot", "many", "saturated"])
def test_host_compiled_replay_matches_the_reference(hostdev, case, loss):
    """The replay's reformulation (k = product^p (bsdfPdf - dTreePdf) / woPdf ahead of the chain, fma in the gradient and the batch sum, beta^iter as
    running double products, iter carried as a float) on every case, compiled for the host: iter and batchAcc exact, m / v / theta / batchGrad within
    the three-sided tolerance, everything finite."""
    states, a, b = make_case(case)
    dut = host_replay(hostdev, states, a, b, loss)
    assert_states(dut, ref32_replay(states, a, b, loss), ref64_replay(states, a, b, loss), (case, loss))


@pytest.mark.parametrize("loss", LOSSES)
def test_host_compiled_replay_of_a_saturated_fraction(hostdev, loss):
    """theta = +20 / +17 (logistic rounds to exactly 1.0f) with dTreePdf > 2^25 bsdfPdf: the reference's mixture is bsdfPdf, its loss term finite x 0 = 0,
    and theta only drifts down under the L2 term, about lr per Adam step.  The replay must do the same: finite, equal to the float32 reference."""
    states, a, b = make_case("saturated")
    dut = host_replay(hostdev, states, a, b, loss); r32 = ref32_replay(states, a, b, loss)
    _assert_saturated(states, dut, r32)


def _l2_only(state, steps):
    """Adam (GP:97-109, float64) on the L2 gradient alone: what theta does when the loss term is finite x f (1 - f) = 0."""
    it, m1, m2, th = int(state[0]), float(state[1]), float(state[2]), float(state[3])
    for _ in range(int(steps)):
        g = 0.01 * th; it += 1
        lr = LR * math.sqrt(1.0 - B2 ** it) / (1.0 - B1 ** it)
        m1 = B1 * m1 + (1.0 - B1) * g; m2 = B2 * m2 + (1.0 - B2) * g * g
        th = min(max(th - lr * m1 / (math.sqrt(m2) + EPS), -20.0), 20.0)
    return th


def _assert_saturated(states, dut, r32):
    assert np.isfinite(dut).all(), dut
    steps = dut[:, 0] - states[:, 0]
    assert (steps > 100).all() and np.array_equal(dut[:, 0], r32[:, 0])
    assert (dut[:, 3] < states[:, 3] - 0.5).all()
    # theta = +20 stays above 17 throughout, so the loss term is 0 at every record: theta follows Adam on the L2 gradient alone (measured: 2e-5 from
    # the float64 walk, the float32 rounding of 200 steps).  The theta = +17 leaves leave saturation after a few steps; the reference comparison covers them.
    sat = states[:, 3] == 20
    l2 = np.array([_l2_only(s, k) for s, k in zip(states[sat], steps[sat])])
    assert sat.sum() == 2 and np.abs(dut[sat, 3] - l2).max() <= 1e-4, (dut[sat, 3], l2)
    assert np.abs(dut[:, 3] - r32[:, 3]).max() <= FLOOR["theta"], (dut[:, 3], r32[:, 3])


# ------------------------------------------------------------------------------------------------------------------- the CUDA kernels
def _gpu_replay(states, a, b, loss, counts=None, **kw):
    from ppg_b200.integrator import op_fraction_replay
    return op_fraction_replay(states, a, b, counts if counts is not None else [[len(a)]], loss, **kw)


def _assert_bucketed(a, b, sa, sb, n_leaves):
    """sa / sb: a permutation of (a, b) bit for bit, each leaf's records contiguous at the exclusive scan of the counts, in input order's multiset."""
    la = leaf_of(a); cnt = np.bincount(la, minlength=n_leaves); off = np.concatenate([[0], np.cumsum(cnt)[:-1]])
    ls = leaf_of(sa)
    assert np.array_equal(ls, np.repeat(np.arange(n_leaves, dtype=np.uint32), cnt))      # contiguous, at offset[leaf]
    key = lambda x, y: np.sort(np.concatenate([x.view(np.uint32), y.view(np.uint32)], axis=1).view(np.dtype((np.void, 24))).ravel())
    assert np.array_equal(key(a, b), key(sa, sb))                                       # a permutation, bit for bit
    return off


def _progress(before, after):
    """adam_progress_kernel recomputed from the states: (sum steps * floor(|f_after - f_before| * 2^20), sum steps, leaves that stepped)."""
    lg = lambda x: np.float32(1) / (np.float32(1) + np.exp(-x.astype(np.float32)))
    ds = after[:, 0] - before[:, 0]; s = ds > 0
    df = np.abs(lg(after[s, 3]) - lg(before[s, 3])).astype(np.float32)
    k = ds[s].astype(np.uint64)
    return int((k * (df * np.float32(1048576.0)).astype(np.uint64)).sum()), int(k.sum()), int(s.sum())


@pytest.mark.gpu
@pytest.mark.parametrize("loss", LOSSES)
@pytest.mark.parametrize("case", ["grid", "hot", "many", "saturated"])
def test_gpu_replay_matches_the_reference(case, loss):
    """adam_hist / exclusive_scan / adam_scatter / adam_seq / adam_progress with the renderer's launch shapes: bucketing exact, then the reference replayed
    in the bucket order the device returned (record for record): iter / batchAcc exact, m / v / theta / batchGrad within the three-sided tolerance, the
    leaf record's theta equal to the state's, the progress counters equal to the kernel's formula on the returned states."""
    states, a, b = make_case(case)
    r = _gpu_replay(states, a, b, loss)
    _assert_bucketed(a, b, r["sorted_a"], r["sorted_b"], len(states))
    dut = r["states"][0]
    r32 = ref32_replay(states, r["sorted_a"], r["sorted_b"], loss); r64 = ref64_replay(states, r["sorted_a"], r["sorted_b"], loss)
    assert_states(dut, r32, r64, (case, loss))
    has = np.bincount(leaf_of(a), minlength=len(states)) > 0                  # adam_seq_kernel writes the leaf record of the leaves it replayed
    assert np.array_equal(r["theta"][0][has], dut[has, 3]) and not r["theta"][0][~has].any() and np.array_equal(dut[~has], states[~has])
    moved, steps, nstep = _progress(states, dut)
    assert int(r["progress"][0, 1]) == steps and abs(int(r["progress"][0, 0]) - moved) <= nstep
    if case == "saturated":
        _assert_saturated(states, dut, r32)


@pytest.mark.gpu
@pytest.mark.parametrize("loss", LOSSES)
def test_gpu_replay_capacity_and_two_batches(loss):
    """A record list shorter than the records appended (only the first `cap` are replayed) and two consecutive batches on the same counting buffers: the
    second batch buckets as if it were the first (adam_seq_kernel reset the counts and cursors), and the replay continues from the first batch's states."""
    states, a, b = make_case("grid", seed=3)
    n = len(a); n1 = n // 2; cap = n1 - 1000
    r = _gpu_replay(states, a, b, loss, counts=[[n1], [n - n1]], cap=cap)
    a1, b1 = a[:cap], b[:cap]; a2, b2 = a[n1:n1 + cap], b[n1:n1 + cap]
    _assert_bucketed(a1, b1, r["sorted_a"][:cap], r["sorted_b"][:cap], len(states))
    _assert_bucketed(a2, b2, r["sorted_a"][n1:n1 + cap], r["sorted_b"][n1:n1 + cap], len(states))
    assert not r["sorted_a"][cap:n1].any() and not r["sorted_a"][n1 + cap:].any()
    prev = states
    for k, (sa, sb) in enumerate(((r["sorted_a"][:cap], r["sorted_b"][:cap]), (r["sorted_a"][n1:n1 + cap], r["sorted_b"][n1:n1 + cap]))):
        dut = r["states"][k]
        assert_states(dut, ref32_replay(prev, sa, sb, loss), ref64_replay(prev, sa, sb, loss), (k, loss))
        moved, steps, nstep = _progress(prev, dut)
        assert int(r["progress"][k, 1]) == steps and abs(int(r["progress"][k, 0]) - moved) <= nstep
        prev = dut


def _merge_rule32(start, reps):
    """adam_pack(1) + the in-order float sum + adam_merge (DESIGN 4.2), emulated in float32 operation by operation."""
    R = len(reps); f = np.float32
    s = np.zeros_like(start)
    for x in reps:
        d = x.copy(); d[:, 0] = x[:, 0] - start[:, 0]
        s = (s + d).astype(np.float32)
    out = np.empty_like(start)
    out[:, 0] = start[:, 0] + s[:, 0]
    out[:, 1:4] = s[:, 1:4] * (f(1) / f(R))
    acc = s[:, 4] - f(R - 1) * start[:, 4]; grad = s[:, 5] - f(R - 1) * start[:, 5]
    out[:, 4] = np.where(acc > 0, acc, f(0)); out[:, 5] = np.where(acc > 0, grad, f(0))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("R", [1, 2, 3, 8])
def test_gpu_replica_merge(R):
    """R replicas replay their own records from the common start, then adam_pack / sum / adam_merge: step counts and batch accumulators add up relative
    to the start, moments and theta are averaged (DESIGN 4.2).  The merged state equals that rule evaluated in float32 in the kernels' order bit for bit,
    and the rule in float64 to the rounding of an R-term float sum; a replica without records leaves the start unchanged; R = 1 merges to the identity."""
    states, a, b = make_case("grid", seed=10 + R)
    rng = np.random.default_rng(R)
    grp = rng.integers(0, R, len(a))
    if R > 1:
        grp[grp == R - 1] = 0                            # the last replica gets no records
    order = np.argsort(grp, kind="stable"); a, b, grp = a[order], b[order], grp[order]
    counts = np.bincount(grp, minlength=R).reshape(1, R)
    r = _gpu_replay(states, a, b, "kl", counts=counts, replicas=R, merge=True)
    reps = r["replicas"][0]
    if R > 1:
        assert np.array_equal(reps[R - 1], states)
    merged = r["states"][0]
    assert np.array_equal(merged.view(np.uint32), _merge_rule32(states, list(reps)).view(np.uint32))
    if R == 1:
        assert np.array_equal(merged, reps[0])
    r64 = reps.astype(np.float64); s64 = states.astype(np.float64)
    ex = np.empty_like(s64)
    ex[:, 0] = s64[:, 0] + (r64[:, :, 0] - s64[:, 0]).sum(0); ex[:, 1:4] = r64[:, :, 1:4].mean(0)
    acc = r64[:, :, 4].sum(0) - (R - 1) * s64[:, 4]
    assert np.array_equal(merged[:, 0], ex[:, 0]) and np.array_equal(merged[:, 4] > 0, acc > 0)
    bound = (R + 1) * np.finfo(np.float32).eps * np.abs(r64[:, :, 1:4]).sum(0) / R + np.spacing(np.abs(ex[:, 1:4]).astype(np.float32))
    assert (np.abs(merged[:, 1:4] - ex[:, 1:4]) <= bound).all()
    assert np.array_equal(r["theta"][0], merged[:, 3])
