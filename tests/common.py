import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def reference_dir():
    """A checkout of the original project (Tom94/practical-path-guiding), for the few checks that need its large scene assets (SPACESHIP 52 MB,
    KITCHEN 140 MB, the Stanford bunny): PPG_REFERENCE_DIR, else the checkout the package reads Mitsuba's data files from
    (ppg_b200.rtrans: <checkout>/mitsuba/data/microfacet).  Those checks skip where neither exists."""
    if os.environ.get("PPG_REFERENCE_DIR"):
        return os.environ["PPG_REFERENCE_DIR"]
    from ppg_b200 import rtrans
    return os.path.dirname(os.path.dirname(os.path.dirname(rtrans._DATA_DIR)))


def reference_file(*parts):
    """Path of a file of the original project's checkout, or None where there is none."""
    p = os.path.join(reference_dir(), *parts)
    return p if os.path.exists(p) else None


def assert_render_parity(img, ref, st, ost, sc=None, props=None, pixels=0.90, mean=0.01, counts=2e-4, leaves=1):
    """Parity of a TRAINED render of the CUDA path (img, st) with the oracle's (ref, ost) on the same seeded inputs.

    Both implementations accumulate the SD-tree statistics with floating-point atomics (the reference's addToAtomicFloat, GP:59-62;
    red.global.add.f32 on the device): the sums differ in the last ulp from run to run, and now and then a path whose random number falls
    between two such roundings of a quadtree partition takes the other child -- from there on the region it trains decorrelates to noise level
    (measured: a handful to a few hundred of 16 384 pixels; a single light-sampled firefly then moves relMSE to 1e-3).  The claim is therefore
    split into a deterministic and a robust part, each checked ONCE (no retry):
      * the unguided first pass (no tree involved) is the same computation on both sides: relMSE <= 1e-9, equal vertex counts
        (checked when `sc` and `props` are given: one extra pass of both implementations; libm ulps flip a discrete decision of a few paths in 10^5);
      * the trained render: total vertices and every iteration's recorded weight within `counts` (2e-4; 2e-3 for the big scenes with rough
        BSDFs, where libm ulps in sincos / pow / erf flip more decisions), leaf counts within `leaves` (1),
        at least `pixels` (90 %) of the pixels equal to 1e-3 relative, the image mean within `mean` (1 %)."""
    if sc is not None:
        import oracle_lib as O
        from ppg_b200.integrator import GuidedPathTracer
        p1 = dict(props, budgetType="spp", budget=props.get("sppPerPass", "4"), sampleCombination="automatic")      # (inversevar weights a one-sample iteration by 1 / inf)
        g = GuidedPathTracer(p1); g.set_scene(sc); i1, s1 = g.render(); g.close()
        o = O.Oracle(O.params_from_xml(p1), sc, kind="port"); r1, os1 = o.render(); o.close()
        assert abs(s1["total_vertices"] - os1["total_vertices"]) <= max(2, 2e-4 * os1["total_vertices"]), (s1["total_vertices"], os1["total_vertices"])
        close1 = np.isclose(i1, r1, rtol=1e-3, atol=1e-5).all(axis=2)
        assert close1.mean() >= 0.998 and relmse(i1[close1], r1[close1]) <= 1e-9, (close1.mean(), relmse(i1, r1))      # (libm ulps may flip a discrete decision of a path or two)
    assert abs(st["total_vertices"] - ost["total_vertices"]) <= max(2, counts * ost["total_vertices"]), (st["total_vertices"], ost["total_vertices"])
    assert len(st["iterations"]) == len(ost["iterations"])
    for a, b in zip(st["iterations"], ost["iterations"]):
        assert a["passes"] == b["passes"] and abs(a["s_tree_leaves"] - b["s_tree_leaves"]) <= leaves, (a["iteration"], a["s_tree_leaves"], b["s_tree_leaves"])
        wa, wb = a["weight_avg"] * a["s_tree_leaves"], b["weight_avg"] * b["s_tree_leaves"]
        assert abs(wa - wb) <= max(4, counts * wb), (a["iteration"], wa, wb)
    close = np.isclose(img, ref, rtol=1e-3, atol=1e-5).all(axis=2)
    assert close.mean() >= pixels, close.mean()
    assert abs(float(img.mean()) - float(ref.mean())) <= mean * float(ref.mean()), (img.mean(), ref.mean())


def load_cbox(size=None, improved=False):
    from ppg_b200.scene import SceneDesc
    sc = SceneDesc.load(os.path.join(ROOT, "scenes", "cbox-improved.npz" if improved else "cbox.npz"))
    if size is not None:
        sc = sc.with_film(size, size)
    return sc


def load_fixture_scene(name, size=None):  # size None or 0: the XML film size
    """scenes/<name>.npz written by tools/make_fixtures.py."""
    from ppg_b200.scene import SceneDesc
    sc = SceneDesc.load(os.path.join(ROOT, "scenes", name + ".npz"))
    return sc.with_film(size, size) if size else sc


def relmse(img, ref):
    img = np.asarray(img, np.float64); ref = np.asarray(ref, np.float64)
    return float(np.mean((img - ref) ** 2 / (ref ** 2 + 1e-3)))


def load_rough_transmittance(dist):
    """Mitsuba's data/microfacet/<dist>.dat as ppg_b200.rtrans.load_table returns it, rebuilt from tests/golden/rough_transmittance_<dist>.npz
    (tools/make_golden.py): the nodes the rough plastics of the tests interpolate; every other node is NaN."""
    z = np.load(os.path.join(ROOT, "tests", "golden", f"rough_transmittance_{dist}.npz"))
    n_eta, n_alpha, n_theta = (int(v) for v in z["shape"])
    trans = np.full((2 * n_eta, n_alpha, n_theta), np.nan, np.float32); diff = np.full((2 * n_eta, n_alpha), np.nan, np.float32)
    trans[z["index"][:, 0], z["index"][:, 1]] = z["trans"]; diff[z["index"][:, 0], z["index"][:, 1]] = z["diff"]
    r = z["ranges"]
    return dict(trans=trans, diff=diff, n_eta=n_eta, n_alpha=n_alpha, n_theta=n_theta, eta_min=r[0], eta_max=r[1], alpha_min=r[2], alpha_max=r[3])


def load_sky_tables():
    """datasetRGB1-3 / datasetRGBRad1-3 of Mitsuba's skymodeldata.h as ppg_b200.sunsky._sky_tables returns them (tests/golden/sky_model_rgb.npz)."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "sky_model_rgb.npz"))
    return {k: z[k] for k in z.files}


def gpu_available():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def cbox_with_sphere(size=128, subdiv=3, center=(185.0, 240.0, 169.0), radius=75.0, smooth=True):
    """CBOX plus a tessellated diffuse sphere (20 * 4^subdiv triangles, smooth vertex normals): more than 64 triangles,
    so the CUDA path intersects through the BVH walk instead of the lock-step tiny-scene test."""
    import copy
    sc = copy.copy(load_cbox(size))
    t = (1.0 + 5 ** 0.5) / 2.0
    v = [(-1, t, 0), (1, t, 0), (-1, -t, 0), (1, -t, 0), (0, -1, t), (0, 1, t), (0, -1, -t), (0, 1, -t), (t, 0, -1), (t, 0, 1), (-t, 0, -1), (-t, 0, 1)]
    f = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6), (7, 1, 8),
         (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10), (8, 6, 7), (9, 8, 1)]
    v = [np.array(p, np.float64) / np.linalg.norm(p) for p in v]
    for _ in range(subdiv):
        cache = {}; nf = []
        def mid(a, b):
            k = (min(a, b), max(a, b))
            if k not in cache:
                m = v[a] + v[b]; v.append(m / np.linalg.norm(m)); cache[k] = len(v) - 1
            return cache[k]
        for a, b, c in f:
            ab, bc, ca = mid(a, b), mid(b, c), mid(c, a)
            nf += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
        f = nf
    V = np.array(v); F = np.array(f, np.uint32)
    P = (np.array(center) + radius * V).astype(np.float32); N = V.astype(np.float32)
    nv, nt, ns = len(sc.positions), len(sc.indices), len(sc.shapes)
    sc.positions = np.concatenate([sc.positions, P]); sc.normals = np.concatenate([sc.normals, N if smooth else np.zeros_like(N)])
    sc.uvs = np.concatenate([sc.uvs, np.zeros((len(P), 2), np.float32)])
    sc.indices = np.concatenate([sc.indices, F + nv]).astype(np.uint32)
    sc.triangle_shape = np.concatenate([sc.triangle_shape, np.full(len(F), ns, np.uint32)])
    sc.shapes = np.concatenate([sc.shapes, np.array([[nt, len(F), 1, -1, 1 if smooth else 0, 0, 0, 0]], np.int32)])   # bsdf 1 = "white"
    return sc
