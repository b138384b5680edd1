"""BSDF restatements of the oracle, checked the way the reference checks its BSDFs (src/tests/test_chisquare.cpp:391-623):
sample() must be distributed according to pdf(), and the sampling weight must equal eval()/pdf()."""
import numpy as np
import pytest

import oracle_lib as O
from reference_outputs import reference

HAVE_MFREF = __import__("os").path.exists(O.MFREF_SO)      # the reference's own functions (oracle/_ref), else the rows stored under tests/golden

CASES = {
    "diffuse": dict(type=0, reflectance=(0.6, 0.5, 0.4)),
    "roughconductor-ggx-0.1": dict(type=4, reflectance=(1, 1, 1), eta=(1.65746, 0.880369, 0.521229), k=(9.22387, 6.26952, 4.837), alpha=0.1, distribution=1),   # spaceship.xml "RoughAluminium"
    "roughconductor-ggx-0.4": dict(type=4, reflectance=(0.9, 0.9, 0.9), eta=(2, 2, 2), k=(0, 0, 0), alpha=0.4, distribution=1),
    "roughdielectric-ggx-0.1": dict(type=6, reflectance=(1, 1, 1), transmittance=(1, 1, 1), eta=(1.5, 1.5, 1.5), alpha=0.1, distribution=1),      # spaceship.xml glass (bk7-like, GGX)
    "roughdielectric-beckmann-0.3": dict(type=6, reflectance=(0.9, 0.8, 1), transmittance=(0.7, 0.9, 1), eta=(1.33, 1.33, 1.33), alpha=0.3, distribution=0),
    "roughdielectric-ggx-0.3-inside": dict(type=6, reflectance=(1, 1, 1), transmittance=(1, 1, 1), eta=(1.5, 1.5, 1.5), alpha=0.3, distribution=1, inside=True),
    "roughconductor-beckmann-0.3": dict(type=4, reflectance=(1, 1, 1), eta=(0.2, 0.9, 1.1), k=(3.9, 2.4, 2.2), alpha=0.3, distribution=0),
}




def _roughplastic(distribution, alpha, nonlinear, diffuse=(0.256, 0.013, 0.08)):
    """(ppg_bsdf, tables) through the host loader's reduction of Mitsuba's data/microfacet tables (rtrans.py; the nodes stored under tests/golden)."""
    from ppg_b200.scene import make_roughplastic
    tables = []
    row = make_roughplastic(0, diffuse, (1, 1, 1), 1.5 / 1.000277, alpha, distribution, nonlinear, tables)
    return O.bsdf_from_row(row), np.asarray(tables, np.float32)


def _plastic(nonlinear, eta):
    from ppg_b200.scene import make_plastic
    return O.bsdf_from_row(make_plastic(0, (0.6, 0.3, 0.2), (1, 1, 1), eta, nonlinear)), None


SMOOTH_PLASTIC = {"plastic-1.49-nonlinear": (True, 1.49), "plastic-1.9": (False, 1.9)}
PLASTIC = {"roughplastic-beckmann-0.4-nonlinear": (0, 0.4, True), "roughplastic-ggx-0.2": (1, 0.2, False), "roughplastic-beckmann-0.1": (0, 0.1, False)}


@pytest.mark.parametrize("name", list(CASES) + list(PLASTIC) + list(SMOOTH_PLASTIC))
@pytest.mark.parametrize("cos_i", [0.95, 0.5, 0.15])
def test_sample_matches_pdf_and_weight_matches_eval(name, cos_i):
    tables = None
    if name in SMOOTH_PLASTIC:
        b, tables = _plastic(*SMOOTH_PLASTIC[name])
    elif name in PLASTIC:
        b, tables = _roughplastic(*PLASTIC[name])
    else:
        kw = dict(CASES[name])
        if kw.pop("inside", False):
            cos_i = -cos_i
        b = O.make_bsdf(**kw)
    _chi2(b, tables, cos_i)


def _chi2(b, tables, cos_i):
    sphere = b.type == 6           # transmissive: histogram over the whole sphere
    rng = np.random.default_rng(1)
    n = 400000
    wi = np.tile(np.array([[np.sqrt(1 - cos_i ** 2), 0.0, cos_i]], np.float32), (n, 1))
    wo, w, pdf, delta = O.bsdf_sample(b, wi, rng.random((n, 2), dtype=np.float32), tables=tables)
    ok = (pdf > 0) & (w.sum(axis=1) > 0) & (delta == 0)         # the smooth part (plastic's coat reflection is a delta lobe)
    assert ok.mean() > 0.2
    if delta.any():       # plastic.cpp:330-340: mirror direction, probability probSpecular, weight specularReflectance * Fi / probSpecular
        dl = delta != 0
        assert np.allclose(wo[dl], wi[dl] * np.float32([-1, -1, 1]), atol=1e-6)
        assert abs(dl.mean() - pdf[dl][0]) < 0.01 and np.allclose(pdf[dl], pdf[dl][0])
    ev, pdf2 = O.bsdf_eval_pdf(b, wi[ok], wo[ok], tables=tables)
    assert np.allclose(pdf2, pdf[ok], rtol=2e-3, atol=1e-6)                       # pdf() of the sampled direction == pdf returned by sample()
    assert np.allclose(ev, w[ok] * pdf[ok, None], rtol=3e-3, atol=1e-5)         # weight == eval / pdf
    # chi^2: histogram of sampled directions vs integral of pdf over a (cos theta, phi) grid on the upper hemisphere
    nb_c, nb_p = (20 if sphere else 10), 20
    lo = -1.0 if sphere else 0.0
    wo_ok = wo[ok]
    ct = np.clip(wo_ok[:, 2], lo, 1); ph = np.mod(np.arctan2(wo_ok[:, 1], wo_ok[:, 0]), 2 * np.pi)
    H, _, _ = np.histogram2d(ct, ph / (2 * np.pi), bins=[nb_c, nb_p], range=[[lo, 1], [0, 1]])
    ng = 32 if sphere else 12      # refraction compresses the lobe: finer quadrature per histogram cell
    g = (np.arange(ng) + 0.5) / ng
    exp = np.zeros((nb_c, nb_p))
    for i in range(nb_c):
        for j in range(nb_p):
            c = (lo + (1 - lo) * (i + g[:, None]) / nb_c + 0 * g[None, :]).ravel(); p = (2 * np.pi * (j + g[None, :]) / nb_p + 0 * g[:, None]).ravel()
            sn = np.sqrt(1 - c * c)
            d = np.stack([sn * np.cos(p), sn * np.sin(p), c], -1).astype(np.float32)
            evq, pd = O.bsdf_eval_pdf(b, np.tile(wi[:1], (len(d), 1)), d, tables=tables)
            if sphere:      # reference quirk kept by the restatement: roughdielectric pdf() is non-zero for grazing refraction configurations whose
                pd = pd * (evq.sum(axis=1) > 0)   # half-vector is unphysical (eval() == 0 through smithG1); sample() never produces them
            exp[i, j] = pd.mean() * ((1 - lo) * 2 * np.pi / (nb_c * nb_p))
    exp *= n                      # failed samples (pdf == 0) carry no mass: compare absolute counts
    mask = exp > 10
    chi2 = np.sum((H[mask] - exp[mask]) ** 2 / exp[mask]); dof = mask.sum() - 1
    assert chi2 < dof + 8 * np.sqrt(2 * dof) + 0.02 * n * 0, (chi2, dof)
    assert abs(H.sum() - exp.sum()) < 0.03 * n


def test_dielectric_and_conductor_are_delta_and_energy_conserving():
    glass = O.make_bsdf(type=2, reflectance=(1, 1, 1), transmittance=(1, 1, 1), eta=(1.5, 1.5, 1.5))
    rng = np.random.default_rng(2)
    n = 100000
    for cz in (0.9, 0.3, -0.6):
        wi = np.tile(np.array([[np.sqrt(1 - cz ** 2), 0, cz]], np.float32), (n, 1))
        wo, w, pdf, delta = O.bsdf_sample(glass, wi, rng.random((n, 2), dtype=np.float32))
        assert delta.all()
        refl = wo[:, 2] * cz > 0
        F = refl.mean()
        assert np.allclose(pdf[refl], F, atol=0.01) and np.allclose(pdf[~refl], 1 - F, atol=0.01)      # discrete lobe probabilities F / 1-F
        assert np.allclose(np.linalg.norm(wo, axis=1), 1, atol=1e-5)
        ev, pd = O.bsdf_eval_pdf(glass, wi, wo)
        assert not ev.any() and not pd.any()                                                           # delta lobes: zero in the solid-angle measure
    mirror = O.make_bsdf(type=3, reflectance=(1, 1, 1), eta=(0, 0, 0), k=(1, 1, 1))
    wi = np.tile(np.array([[0.6, 0, 0.8]], np.float32), (4, 1))
    wo, w, pdf, delta = O.bsdf_sample(mirror, wi, rng.random((4, 2), dtype=np.float32))
    assert np.allclose(wo, [-0.6, 0, 0.8]) and np.allclose(w, 1.0, atol=1e-5) and np.allclose(pdf, 1) and delta.all()   # eta=0,k=1: perfect mirror (conductor.cpp:159-176)


def test_thin_dielectric_folds_internal_reflections_and_transmits_straight():
    """thindielectric.cpp:206-240: reflection with probability R' = R + T^2 R / (1 - R^2), else the ray goes straight through (ENull)."""
    b = O.make_bsdf(type=8, reflectance=(1, 1, 1), transmittance=(0.8, 0.9, 1.0), eta=(1.5, 1.5, 1.5))
    rng = np.random.default_rng(3)
    n = 200000
    for cz in (0.9, 0.2, -0.5):
        wi = np.tile(np.array([[np.sqrt(1 - cz ** 2), 0, cz]], np.float32), (n, 1))
        wo, w, pdf, delta = O.bsdf_sample(b, wi, rng.random((n, 2), dtype=np.float32))
        assert delta.all()
        refl = wo[:, 2] * cz > 0
        c = abs(cz); ct = np.sqrt(1 - (1 - c * c) / 2.25)
        R = 0.5 * (((c - 1.5 * ct) / (c + 1.5 * ct)) ** 2 + ((1.5 * c - ct) / (1.5 * c + ct)) ** 2); Rp = R + (1 - R) ** 2 * R / (1 - R * R)
        assert abs(refl.mean() - Rp) < 0.005 and np.allclose(pdf[refl], Rp, atol=1e-5) and np.allclose(pdf[~refl], 1 - Rp, atol=1e-5)
        assert np.allclose(wo[~refl], -wi[~refl], atol=1e-7) and np.allclose(wo[refl], wi[refl] * np.float32([-1, -1, 1]), atol=1e-7)
        assert np.allclose(w[~refl], [0.8, 0.9, 1.0]) and np.allclose(w[refl], 1.0)


def test_oracle_looks_through_null_surfaces_consistently():
    """With every light path crossing an index-matched pane, BSDF sampling alone (nee=never: emitter lookup through the pane) and the
    plain CBOX bracket the result; light sampling adds the reference's known excess (MIS pdf from the last segment only, GP:2236 +
    records.inl:170-178) -- both facts pinned here so that a change of either code path is noticed."""
    from common import load_cbox
    from ppg_b200.builtin_scenes import cbox_thin_glass
    base = load_cbox(48); sc = cbox_thin_glass(base)
    mean = {}
    for name, scene, nee in (("plain", base, "never"), ("never", sc, "never"), ("always", sc, "always")):
        o = O.Oracle(O.params_from_xml(dict(scene.integrator, budget="252", nee=nee)), scene, kind="port"); img, st = o.render()
        assert np.isfinite(img).all(); mean[name] = float(img.mean())
    assert 0.85 * mean["plain"] < mean["never"] < mean["plain"]
    assert 1.1 * mean["never"] < mean["always"] < 1.6 * mean["never"]


@pytest.mark.parametrize("type_", [0, 1])          # PPG_MICROFACET_BECKMANN, PPG_MICROFACET_GGX
@pytest.mark.parametrize("alpha", [0.01, 0.1, 0.2, 0.6])
def test_restated_microfacet_equals_the_reference_class(type_, alpha):
    """The oracle's microfacet restatement (struct Microfacet of ppg_cpu_tracer.h: D, Smith G1, the Heitz-d'Eon visible-normal sampling with its Newton
    iteration / rational fits, and mts_erf / mts_erfinv) against the reference's OWN class MicrofacetDistribution (src/bsdfs/microfacet.h:45-721) and math::erf /
    erfinv (src/libcore/math.cpp:25-72) compiled verbatim: same inputs, every float must agree bit for bit (both sides are built without FMA contraction and
    call the same libm).  This is what roughconductor / roughplastic / roughdielectric are built on -- and what the CUDA mf_* functions mirror.
    Without oracle/_ref the reference's outputs are the rows stored under tests/golden (tests/reference_outputs.py)."""
    ref, port = (O.microfacet("ref") if HAVE_MFREF else None), O.microfacet("port")
    live = lambda f: f if HAVE_MFREF else None
    key = f"microfacet/{type_}/{alpha}"
    rng = np.random.default_rng(100 * type_ + int(alpha * 100))
    n = 200000
    def dirs(upper):
        d = rng.normal(size=(n, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
        if upper:
            d[:, 2] = np.abs(d[:, 2])
        return d.astype(np.float32)
    m, v, wi = dirs(False), dirs(False), dirs(True)
    # grazing and near-normal incidence, where the sampling code switches branches (theta < 1e-4, cot / tan extremes)
    wi[:1000] = [0, 0, 1]; wi[1000:2000, 2] = 1e-3 * rng.random(1000); wi[1000:2000] /= np.linalg.norm(wi[1000:2000], axis=1, keepdims=True)
    ma = np.abs(m)
    i, (e, g, p) = reference(key, live(lambda: [ref.eval(type_, alpha, m), ref.smith_g1(type_, alpha, v, m), ref.pdf(type_, alpha, wi, ma)]), n)
    assert np.array_equal(e, port.eval(type_, alpha, m[i]))
    assert np.array_equal(g, port.smith_g1(type_, alpha, v[i], m[i]))
    assert np.array_equal(p, port.pdf(type_, alpha, wi[i], ma[i]))
    smp = rng.random((n, 2), dtype=np.float32); smp[:50] = [[0.0, 0.0]] * 50; smp[50:100] = [[0.99999994, 0.99999994]] * 50
    i, (mr, pr) = reference(key + "/sample", live(lambda: ref.sample(type_, alpha, wi, smp)), n)
    _, (ok_frac,) = reference(key + "/sample_finite", live(lambda: [np.array([np.isfinite(ref.sample(type_, alpha, wi, smp)[0]).all(axis=1).mean()])]), 1)
    mp, pp = port.sample(type_, alpha, wi[i], smp[i])
    ok = np.isfinite(mr).all(axis=1)
    assert ok_frac[0] > 0.999 and np.array_equal(np.isfinite(mp).all(axis=1), ok)
    assert np.array_equal(mr[ok], mp[ok]) and np.array_equal(pr[ok], pp[ok])
    x = np.concatenate([rng.uniform(-0.999999, 0.999999, 100000), [-0.99999994, 0.0, 0.99999994], rng.uniform(-6, 6, 1000)]).astype(np.float32)
    i, (er, eir) = reference(key + "/erf", live(lambda: ref.erf(x)), len(x))
    ep, eip = port.erf(x[i]); inside = np.abs(x[i]) < 1
    assert np.array_equal(er, ep) and np.array_equal(eir[inside], eip[inside])


def test_restated_helpers_equal_the_reference_functions():
    """fresnelDielectricExt, the Spectrum overload of fresnelConductorExact, coordinateSystem (src/libcore/util.cpp:592-601, 651-681, 739-761) and
    warp::squareToCosineHemisphere (warp.cpp:43-52, 81-102), compiled verbatim, against the oracle's restatements: bit for bit."""
    ref, port = (O.microfacet("ref") if HAVE_MFREF else None), O.microfacet("port")
    live = lambda f: f if HAVE_MFREF else None
    rng = np.random.default_rng(9)
    c = np.concatenate([rng.uniform(-1, 1, 200000), [0.0, 1.0, -1.0, 1e-6, -1e-6]]).astype(np.float32)
    for eta in (1.0, 1.5046 / 1.000277, 1 / 1.5, 1.33, 2.4):
        i, (fr, tr) = reference(f"fresnel_dielectric_ext/{eta:.6f}", live(lambda: ref.fresnel_dielectric_ext(c, eta)), len(c))
        fp, tp = port.fresnel_dielectric_ext(c[i], eta)
        assert np.array_equal(fr, fp) and np.array_equal(tr, tp)
    for eta, k in (((0.2, 0.9, 1.1), (3.9, 2.4, 2.2)), ((1.65746, 0.880369, 0.521229), (9.22387, 6.26952, 4.837)), ((0, 0, 0), (1, 1, 1)), ((1.5, 1.5, 1.5), (0, 0, 0))):
        i, (fc,) = reference(f"fresnel_conductor_exact/{eta[0]}/{k[0]}", live(lambda: [ref.fresnel_conductor_exact(np.abs(c), eta, k)]), len(c))
        assert np.array_equal(fc, port.fresnel_conductor_exact(np.abs(c[i]), eta, k))
    a = rng.normal(size=(200000, 3)).astype(np.float32); a /= np.linalg.norm(a, axis=1, keepdims=True); a[:3] = np.eye(3)
    i, (br, cr) = reference("coordinate_system", live(lambda: ref.coordinate_system(a)), len(a))
    bp, cp = port.coordinate_system(a[i])
    assert np.array_equal(br, bp) and np.array_equal(cr, cp)
    smp = rng.random((200000, 2), dtype=np.float32); smp[:4] = [[0.5, 0.5], [0, 0], [0.99999994, 0.5], [0.5, 0]]
    i, (wr,) = reference("square_to_cosine_hemisphere", live(lambda: [ref.square_to_cosine_hemisphere(smp)]), len(smp))
    assert np.array_equal(wr, port.square_to_cosine_hemisphere(smp[i]))


def test_restated_triangle_test_and_spline_equal_the_reference():
    """struct TriAccel (include/mitsuba/render/triaccel.h: Wald's precomputation `load` and `rayIntersect`) and evalCubicInterp1D (src/libcore/spline.cpp:23-60, the
    rough-transmittance lookup of roughplastic), compiled verbatim, against triaccel_load / triaccel_intersect / rough_transmittance of the oracle: the projection axis, the
    nine constants, the hit decision and (t, u, v) agree bit for bit -- the numbers every intersection of oracle and CUDA path (same operations) starts from."""
    import ctypes as C
    ref = C.CDLL(O.MFREF_SO) if HAVE_MFREF else None; port = O.load("port")
    live = lambda f: f if HAVE_MFREF else None
    f32p = C.POINTER(C.c_float)
    rng = np.random.default_rng(21)
    n = 300000
    A = rng.normal(size=(n, 3)).astype(np.float32) * 10; B = A + rng.normal(size=(n, 3)).astype(np.float32); Cc = A + rng.normal(size=(n, 3)).astype(np.float32)
    A[:100, 0] = 0; B[:100, 0] = 0; Cc[:100, 0] = 0                                  # axis-aligned triangles (k = 0 with exact zeros)
    B[100:200] = A[100:200]                                                           # degenerate: denom == 0 -> k = 3, never hit
    # rays aimed at a point near the triangle (about a quarter hit), some parallel to the plane
    w = rng.random((n, 2)); tgt = A + (B - A) * (w[:, :1] * 1.4 - 0.2) + (Cc - A) * (w[:, 1:] * 1.4 - 0.2)
    o = (tgt + rng.normal(size=(n, 3)) * 5).astype(np.float32); d = (tgt - o); d /= np.linalg.norm(d, axis=1, keepdims=True); d = d.astype(np.float32)
    d[200:300] = (B - A)[200:300] / np.linalg.norm((B - A)[200:300], axis=1, keepdims=True)
    mint = np.full(n, 1e-4, np.float32); maxt = np.where(rng.random(n) < 0.1, 3.0, np.inf).astype(np.float32)
    def run(lib, name, sel):
        args = [np.ascontiguousarray(a[sel], np.float32) for a in (A, B, Cc, o, d, mint, maxt)]; m = len(args[0])
        k = np.zeros(m, np.int32); c9 = np.zeros((m, 9), np.float32); hit = np.zeros(m, np.uint8); tuv = np.zeros((m, 3), np.float32)
        fn = getattr(lib, name); fn.argtypes = [C.c_size_t] + [f32p] * 7 + [C.POINTER(C.c_int), f32p, C.POINTER(C.c_ubyte), f32p]
        fn(m, *[a.ctypes.data_as(f32p) for a in args], k.ctypes.data_as(C.POINTER(C.c_int)), c9.ctypes.data_as(f32p), hit.ctypes.data_as(C.POINTER(C.c_ubyte)), tuv.ctypes.data_as(f32p))
        return k, c9, hit, tuv
    i, (k0, c0, h0, t0) = reference("triaccel", live(lambda: run(ref, "mfref_triaccel", slice(None))), n)
    k1, c1, h1, t1 = run(port, "ppgo_triaccel", i)
    assert np.array_equal(k0, k1) and (k0[(i >= 100) & (i < 200)] == 3).all() and 0.1 < h0.mean() < 0.5
    ok = k0 < 3
    assert np.array_equal(c0[ok].view(np.uint32), c1[ok].view(np.uint32))             # (bit patterns: NaN-free here, and -0.0 must stay -0.0)
    assert np.array_equal(h0, h1) and np.array_equal(t0[h0 == 1], t1[h0 == 1])
    # spline: the 100-entry transmittance table of a material, looked up at |cos|^(1/4) and clamped to [0, 1] (rtrans.h:183-193, 233)
    from ppg_b200 import rtrans
    lut, _ = rtrans.reduce_for_material("ggx", 1.5, 0.2)
    lut = np.ascontiguousarray(lut, np.float32)
    cs = np.concatenate([rng.random(100000), [0.0, 1.0, 1e-8]]).astype(np.float32)
    port.ppgo_rough_transmittance.argtypes = [C.c_size_t, f32p, f32p, f32p]
    x = np.power(np.abs(cs), np.float32(0.25)).astype(np.float32)
    def spline():
        a = np.zeros_like(cs)
        ref.mfref_cubic_interp_1d.argtypes = [C.c_size_t, f32p, f32p, C.c_size_t, C.c_float, C.c_float, f32p]
        ref.mfref_cubic_interp_1d(len(cs), x.ctypes.data_as(f32p), lut.ctypes.data_as(f32p), len(lut), 0.0, 1.0, a.ctypes.data_as(f32p))
        return [a]
    i, (a,) = reference("cubic_interp_1d", live(spline), len(cs))
    csi = np.ascontiguousarray(cs[i]); b = np.zeros_like(csi)
    port.ppgo_rough_transmittance(len(csi), csi.ctypes.data_as(f32p), lut.ctypes.data_as(f32p), b.ctypes.data_as(f32p))
    # (the abscissa |cos|^(1/4) is computed by numpy for the reference function and by libm's powf inside the restatement: equal in most cases, one ulp apart otherwise)
    assert np.abs(np.clip(a, 0, 1) - b).max() <= 2e-6 and (np.clip(a, 0, 1) == b).mean() > 0.9


def test_restated_discrete_distribution_equals_the_reference():
    """struct DiscreteDistribution (include/mitsuba/core/pmf.h:35-210: append, normalize, sample, sampleReuse), compiled verbatim, against the cumulative tables the
    oracle's light sampling builds and Scene::cdfSample: the normalised entries, the sum, the chosen index and the reused sample agree bit for bit -- with zero-weight
    entries (which `sample` skips), a dominant entry and samples on the table's own boundaries."""
    import ctypes as C
    ref = C.CDLL(O.MFREF_SO) if HAVE_MFREF else None; port = O.load("port")
    live = lambda f: f if HAVE_MFREF else None
    f32p = C.POINTER(C.c_float); u32p = C.POINTER(C.c_uint32)
    rng = np.random.default_rng(33)
    for ne in (1, 2, 7, 300):
        w = rng.lognormal(0, 2, ne).astype(np.float32)
        if ne > 2:
            w[rng.integers(0, ne, max(1, ne // 5))] = 0; w[0] = 0; w[-1] = 0
        w[ne // 2] = max(w[ne // 2], 1e-3)
        n = 100000
        smp = rng.random(n, dtype=np.float32)
        cdf = np.concatenate([[0], np.cumsum(w, dtype=np.float32)]); smp[:ne + 1] = np.minimum(cdf / cdf[-1], np.float32(0.99999994))     # boundaries (approximately: float32 cumsum)
        smp[ne + 1] = 0.0
        def run(lib, name, sel):
            x = np.ascontiguousarray(smp[sel]); m = len(x)
            pdf = np.zeros(ne, np.float32); s = C.c_float(); idx = np.zeros(m, np.uint32); reuse = np.zeros(m, np.float32)
            fn = getattr(lib, name); fn.argtypes = [C.c_size_t, f32p, C.c_size_t, f32p, f32p, C.POINTER(C.c_float), u32p, f32p]
            fn(ne, w.ctypes.data_as(f32p), m, x.ctypes.data_as(f32p), pdf.ctypes.data_as(f32p), C.byref(s), idx.ctypes.data_as(u32p), reuse.ctypes.data_as(f32p))
            return pdf, np.array([s.value], np.float32), idx, reuse
        j, (p0,) = reference(f"discrete/{ne}/pdf", live(lambda: run(ref, "mfref_discrete", slice(None))[:1]), ne)
        _, (s0,) = reference(f"discrete/{ne}/sum", live(lambda: run(ref, "mfref_discrete", slice(None))[1:2]), 1)
        i, (i0, r0) = reference(f"discrete/{ne}/sample", live(lambda: run(ref, "mfref_discrete", slice(None))[2:]), n)
        p1, s1, i1, r1 = run(port, "ppgo_discrete", i)
        assert np.array_equal(p0, p1[j]) and s0 == s1 and np.array_equal(i0, i1) and np.array_equal(r0.view(np.uint32), r1.view(np.uint32)), ne
        assert (w[i0] > 0).all()                                                   # an entry of probability 0 is never returned (pmf.h:131-134)
