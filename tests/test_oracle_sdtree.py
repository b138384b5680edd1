"""Pins the restated SD-tree (oracle/sdtree_port.h) against the reference's OWN SD-tree code compiled verbatim
(oracle/_ref/libppg_oracle_ref.so, built from guided_path.cpp:25-1008 where the original project is present; without it, against the
digests of the reference's results stored under tests/golden).  Single-threaded, same record order -> every float must agree bit for bit."""
import os
import shutil

import numpy as np
import pytest

import oracle_lib as O
from common import ROOT
from reference_outputs import digest, reference_digests

AABB = ([0.0, 0.0, -800.0], [556.0, 548.8, 559.2])


def _records(n, seed):
    rng = np.random.default_rng(seed)
    pos = (rng.random((n, 3)) * np.array([556, 548.8, 559.2])).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32); d /= np.linalg.norm(d, axis=1, keepdims=True)
    rad = rng.lognormal(0, 1, n).astype(np.float32)
    prod = (rad * rng.random(n)).astype(np.float32)
    wo = (0.05 + rng.random(n)).astype(np.float32); bp = (0.05 + rng.random(n)).astype(np.float32); dp = (0.05 + rng.random(n)).astype(np.float32)
    rnd = rng.random((n, 3)).astype(np.float32)
    delta = (rng.random(n) < 0.05).astype(np.uint8)
    return pos, d, rad, prod, wo, bp, dp, rnd, delta


def _run(kind, sfilter, dfilter, loss, iters=3, n=6000):
    o = O.Oracle(O.default_params(), aabb=AABB, kind=kind)
    out = []
    for it in range(iters):
        o.refine(int(np.sqrt(2 ** it) * 300)); o.reset(20, 0.01)
        pos, d, rad, prod, wo, bp, dp, rnd, delta = _records(n * 2 ** it, 100 + it)
        o.record(pos, d, rad, wo, product=prod, bsdf_pdf=bp, dtree_pdf=dp, weight=np.ones(len(rad), np.float32), is_delta=delta, rnd=rnd,
                 sfilter=sfilter, dfilter=dfilter, loss=loss if it > 0 else 0)
        out.append(o.export(1))
        o.build()
        out.append(o.export(0))
    return o, out


@pytest.mark.parametrize("sfilter,dfilter,loss", [(0, 0, 0), (1, 1, 1), (2, 1, 2), (2, 0, 0)])
def test_port_equals_verbatim_reference(sfilter, dfilter, loss):
    def results(kind):
        """Every exported tree array after each refine / record and build, then sample / pdf / lookup / sampling fraction on the trained trees."""
        o, ex = _run(kind, sfilter, dfilter, loss)
        out = {f"{i}/{k}": e[k] for i, e in enumerate(ex) for k in ("s_children", "s_axis", "s_is_leaf", "tree_first", "tree_count", "tree_depth", "children",
                                                                        "tree_sum", "tree_weight", "sums", "adam", "aabb")}
        rng = np.random.default_rng(5)
        e = ex[-1]
        leaves = np.nonzero(e["s_is_leaf"])[0].astype(np.uint32)
        ql = rng.choice(leaves, 20000).astype(np.uint32)
        d = rng.normal(size=(20000, 3)).astype(np.float32); d /= np.linalg.norm(d, axis=1, keepdims=True)
        out["pdf"] = o.pdf(ql, d)
        out["sample"] = o.sample(ql, rng.random((20000, 48), dtype=np.float32))
        pts = (rng.random((20000, 3)) * np.array([556, 548.8, 1359.2]) + np.array([0, 0, -800])).astype(np.float32)
        out["lookup_leaf"], out["lookup_size"] = o.lookup(pts)
        out["fraction"] = o.fraction(leaves)
        return out
    ref = reference_digests(f"sdtree/{sfilter}/{dfilter}/{loss}", (lambda: results("ref")) if O.have_ref() else None)
    port = results("port")
    assert set(port) == set(ref)
    for k in sorted(port, key=lambda k: (len(k), k)):
        assert digest(port[k]) == ref[k], k                 # bit exact


def test_initial_tree_is_uniform_depth_4():
    """DTree::reset with total == 0 refines by 0.25^depth > 0.01 -> depth 4, 85 nodes (GP:484-487; log 'Node count = 85')."""
    o = O.Oracle(O.default_params(), aabb=AABB)
    o.reset(20, 0.01)
    e = o.export(1)
    assert e["tree_count"][0] == 85 and e["tree_depth"][0] == 4 and e["n_leaves"] == 1


def test_empty_tree_pdf_is_uniform_and_sample_is_identity():
    o = O.Oracle(O.default_params(), aabb=AABB)
    o.reset(20, 0.01); o.build()
    d = np.array([[0, 0, 1], [1, 0, 0], [0.6, 0, 0.8]], np.float32)
    assert np.allclose(o.pdf(np.zeros(3, np.uint32), d), 1 / (4 * np.pi))
    rnd = np.array([[0.25, 0.5] + [0] * 6], np.float32)
    got = o.sample(np.zeros(1, np.uint32), rnd)[0]
    ct = 2 * 0.25 - 1; st = np.sqrt(1 - ct * ct)
    assert np.allclose(got, [st * np.cos(np.pi), st * np.sin(np.pi), ct], atol=1e-6)


def test_refine_threshold_and_weight_halving():
    """A leaf splits while its building weight exceeds the threshold; children get half (GP:953-955, 886-892)."""
    o = O.Oracle(O.default_params(), aabb=AABB)
    o.reset(20, 0.01)
    n = 1000
    pos, d, rad, prod, wo, *_ = _records(n, 1)
    o.record(pos, d, rad, wo, weight=np.ones(n, np.float32))
    o.build()
    o.refine(100)       # 1000 -> 500 -> 250 -> 125 -> 62.5: 4 levels, 16 leaves
    e = o.export(1)
    assert e["n_leaves"] == 16
    assert np.allclose(e["tree_weight"][e["s_is_leaf"] == 1], 62.5)


def test_dtree_sample_matches_pdf_chi2():
    """chi^2-style check in the spirit of the reference's test_chisquare.cpp: the histogram of D-tree samples
    matches the integral of D-tree pdf over a 16x32 (cos theta, phi) grid."""
    o = O.Oracle(O.default_params(), aabb=AABB)
    o.reset(20, 0.01)
    rng = np.random.default_rng(2)
    n = 50000
    d = rng.normal(size=(n, 3)); d[:, 2] = np.abs(d[:, 2]) * 2 + 0.5; d /= np.linalg.norm(d, axis=1, keepdims=True)
    pos = np.tile(np.array([[100, 100, 100]], np.float32), (n, 1))
    o.record(pos, d.astype(np.float32), rng.lognormal(0, 0.5, n).astype(np.float32), np.full(n, 0.3, np.float32), weight=np.ones(n, np.float32))
    o.build(); o.reset(20, 0.01)
    o.record(pos, d.astype(np.float32), rng.lognormal(0, 0.5, n).astype(np.float32), np.full(n, 0.3, np.float32), weight=np.ones(n, np.float32))
    o.build()
    m = 400000
    s = o.sample(np.zeros(m, np.uint32), rng.random((m, 48), dtype=np.float32))
    ct = np.clip(s[:, 2], -1, 1); phi = np.mod(np.arctan2(s[:, 1], s[:, 0]), 2 * np.pi)
    H, _, _ = np.histogram2d((ct + 1) / 2, phi / (2 * np.pi), bins=[16, 32], range=[[0, 1], [0, 1]])
    # expected: integrate pdf over each cell with a 8x8 midpoint rule (solid angle of a cell = 4 pi / (16*32))
    g = (np.arange(8) + 0.5) / 8
    exp = np.zeros((16, 32))
    for i in range(16):
        for j in range(32):
            x = (i + g[:, None]) / 16 + 0 * g[None, :]; y = (j + g[None, :]) / 32 + 0 * g[:, None]
            c = 2 * x - 1; sn = np.sqrt(1 - c * c); ph = 2 * np.pi * y
            dirs = np.stack([sn * np.cos(ph), sn * np.sin(ph), c], -1).reshape(-1, 3).astype(np.float32)
            exp[i, j] = o.pdf(np.zeros(64, np.uint32), dirs).mean() * 4 * np.pi / (16 * 32)
    exp *= m
    mask = exp > 5
    chi2 = np.sum((H[mask] - exp[mask]) ** 2 / exp[mask])
    dof = mask.sum() - 1
    assert chi2 < dof + 6 * np.sqrt(2 * dof), (chi2, dof)
    assert abs(H[~mask].sum() - exp[~mask].sum()) < 0.01 * m


SDT_GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_tree-02.sdt")
SDT_CAM = np.arange(16, dtype=np.float32).reshape(4, 4) * 0.25 - 1


def test_sdt_reader_reads_what_the_reference_writes(tmp_path):
    """The .sdt wire format (SURVEY 8f row 2), pinned on the reference's OWN writer: the verbatim BlobWriter / STree::dump / DTree::dump code (GP:35-57, 945-951,
    699-711) dumps a trained tree, ppg_b200.sdt.read (the reader of the visualizer, main.cpp:142-173, restated) reads it back: the camera matrix, one record
    per leaf with sampling weight > 0 in depth-first order, min corner / size of the leaf's voxel, mean, weight, and the node arrays bit for bit.
    Without oracle/_ref the file is the one the reference wrote for this run (tests/golden/reference_tree-02.sdt, tools/make_golden.py) and the trees it
    is read against are the restated ones, bit-equal to the reference's (test_port_equals_verbatim_reference)."""
    from ppg_b200 import sdt
    o, _ = _run("ref" if O.have_ref() else "port", 2, 1, 0, iters=3, n=4000)
    cam = SDT_CAM
    path = tmp_path / "tree-02.sdt"
    if O.have_ref():
        assert o.dump(path, cam) == 0
        assert path.read_bytes() == open(SDT_GOLDEN, "rb").read(), "the stored .sdt file is stale (tools/make_golden.py)"
    else:
        shutil.copyfile(SDT_GOLDEN, path)
    cam2, leaves = sdt.read(path)
    assert np.array_equal(cam2, cam)
    e = o.export(0)                                                                 # the sampling trees the dump holds
    # depth-first order over the S-tree (child 0 first), voxels from the box: the reference dumps leaves with weight > 0 only
    lo, hi = np.float32(AABB[0]), np.float32(AABB[1])
    ext = np.float32(hi - lo); ext[:] = ext.max()                                   # STree::STree cubifies the box from the min corner (GP:850-860)
    order = []
    def walk(n, p, s):
        if e["s_is_leaf"][n]:
            order.append((n, p.copy(), s.copy())); return
        ax = int(e["s_axis"][n]); s2 = s.copy(); s2[ax] = s2[ax] / 2
        walk(int(e["s_children"][n, 0]), p, s2)
        p2 = p.copy(); p2[ax] += s2[ax]
        walk(int(e["s_children"][n, 1]), p2, s2)
    walk(0, lo.copy(), ext.copy())
    kept = [(n, p, s) for n, p, s in order if e["tree_weight"][n] > 0]
    assert len(leaves) == len(kept) > 4
    for leaf, (n, p, s) in zip(leaves, kept):
        f, c = int(e["tree_first"][n]), int(e["tree_count"][n])
        assert np.array_equal(leaf.sums, e["sums"][f:f + c]) and np.array_equal(leaf.children, e["children"][f:f + c])
        assert np.allclose(leaf.pos, p, rtol=1e-6, atol=1e-4) and np.allclose(leaf.size, s, rtol=1e-6)
        assert leaf.weight == int(e["tree_weight"][n]) and leaf.depth() == int(e["tree_depth"][n])
        w = float(e["tree_weight"][n])
        assert np.isclose(leaf.mean, float(e["tree_sum"][n]) / (4 * np.pi * w), rtol=1e-5)
    # the density the reader reconstructs is the density the reference samples with
    rng = np.random.default_rng(1)
    d = rng.normal(size=(200, 3)).astype(np.float32); d /= np.linalg.norm(d, axis=1, keepdims=True)
    n0 = kept[0][0]
    ref = o.pdf(np.full(len(d), n0, np.uint32), d)
    xy = np.stack([(np.clip(d[:, 2], -1, 1) + 1) / 2, np.mod(np.arctan2(d[:, 1], d[:, 0]), 2 * np.pi) / (2 * np.pi)], 1)      # dirToCanonical, GP:597-608
    mine = np.array([leaves[0].pdf(float(x), float(y)) for x, y in xy])
    assert np.allclose(mine, ref, rtol=1e-4, atol=1e-7)
    # and a damaged file is an error, not a guess
    raw = open(path, "rb").read(); (tmp_path / "cut.sdt").write_bytes(raw[:len(raw) - 7])
    with pytest.raises(ValueError):
        sdt.read(tmp_path / "cut.sdt")
    assert O.Oracle(O.default_params(), aabb=AABB, kind="port").dump(tmp_path / "x.sdt", cam) == -6      # the restated backend has no writer of its own


@pytest.mark.parametrize("sfilter,dfilter,loss", [(0, 0, 0), (1, 1, 1), (2, 1, 2), (1, 0, 0), (2, 0, 1)])
def test_restated_commit_equals_the_reference_vertex_commit(sfilter, dfilter, loss):
    """Vertex::commit (GP:1730-1768) -- validity test, radiance / throughput per channel above Epsilon, the product with the BSDF value, channel averages, the
    spatial filters (nearest / stochastic with its three jitter numbers and the clip to the scene box / box) -- in the reference's OWN struct Vertex, compiled
    verbatim into oracle/_ref, against the restated commit_vertex of the tracer: the same vertices, committed in the same order, must leave the same trees
    bit for bit -- on the reference's trees and on the restated trees."""
    rng = np.random.default_rng(40 + sfilter * 9 + dfilter * 3 + loss)
    trees = {"verbatim": O.Oracle(O.default_params(), aabb=AABB, kind="ref"), "restated on ref trees": O.Oracle(O.default_params(), aabb=AABB, kind="ref"),
             "restated on port trees": O.Oracle(O.default_params(), aabb=AABB, kind="port")} if O.have_ref() else \
        {"restated on port trees": O.Oracle(O.default_params(), aabb=AABB, kind="port")}          # without oracle/_ref: the verbatim trees' digests
    verbatim = {}
    for it in range(3):
        n = 5000 * 2 ** it
        pos, d, rad, prod, wo, bp, dp, rnd, delta = _records(n, 300 + it)
        thr = (rng.lognormal(-1, 1.5, (n, 3))).astype(np.float32); bv = rng.random((n, 3)).astype(np.float32)
        radiance = (thr * rng.lognormal(0, 1, (n, 3))).astype(np.float32)
        # the cases the early return and the per-channel guard exist for
        radiance[::97, 0] = np.nan; radiance[::89, 1] = -1.0; bv[::83, 2] = np.inf; wo[::79] = 0.0; wo[::73] = -0.5
        thr[::71, 0] = 1e-6; thr[::67] = 0.0; thr[::61, 2] = 3e-5
        weight = np.where(rng.random(n) < 0.3, 0.5, 1.0).astype(np.float32)
        for name, o in trees.items():
            o.refine(int(np.sqrt(2 ** it) * 300)); o.reset(20, 0.01)
            assert o.commit(pos, d, thr, bv, radiance, wo, bp, dp, weight, delta, rnd, sfilter, dfilter, loss if it > 0 else 0, verbatim=(name == "verbatim")) == 0
        ex = {name: o.export(1) for name, o in trees.items()}
        keys = ("sums", "children", "tree_weight", "tree_sum", "adam", "s_children")
        verbatim[it] = reference_digests(f"commit/{sfilter}/{dfilter}/{loss}/{it}", (lambda: {key: ex["verbatim"][key] for key in keys}) if O.have_ref() else None)
        for key in keys:
            for name in ex:
                if name != "verbatim":
                    assert digest(ex[name][key]) == verbatim[it][key], (it, key, name)
        assert ex["restated on port trees"]["tree_weight"].sum() > 0.1 * n          # (the box filter spreads a record over the overlapped leaves by volume)
        for o in trees.values():
            o.build()
    assert trees["restated on port trees"].commit(pos, d, thr, bv, radiance, wo, bp, dp, weight, delta, rnd, verbatim=True) == -6      # no reference code in the restated build
