"""The product's CUDA device functions (practical-path-guiding_b200/csrc/ppg_device.cuh) compiled for the HOST with g++ (tests/hostdev/: CUDA's own headers supply
float3 / float4, the intrinsics get host meanings) and compared, function by function and bit for bit, with the reference's own code compiled verbatim
(oracle/_ref/libmicrofacet_ref.so) -- or with the oracle's restatement where the reference tree was absent at build time.  The kernels are built with -fmad=false
-prec-div=true -prec-sqrt=true, this harness with -ffp-contract=off: +, -, *, / and sqrt round identically; only the libm calls are the host's here and the
device's on the GPU (their ulps are what the `-m gpu` parity tests allow for).  So: reference source == oracle == the source the kernels are compiled from."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle_lib as O
from common import ROOT

CUDA_INC = next((p for p in (os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include"), "/usr/local/cuda/include") if os.path.exists(os.path.join(p, "cuda_runtime.h"))), None)
pytestmark = pytest.mark.skipif(CUDA_INC is None or shutil.which("g++") is None, reason="needs g++ and the CUDA headers")
f32p = C.POINTER(C.c_float)


@pytest.fixture(scope="module")
def dev(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("hostdev") / "libdevice_on_host.so")
    cmd = ["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I" + CUDA_INC, "-D__device__=", "-D__host__=", "-D__global__=", "-D__shared__=",
           "-D__forceinline__=inline", "-D__noinline__=", "-D__launch_bounds__(...)=", "-Wno-unused-function", os.path.join(ROOT, "tests", "hostdev", "device_on_host.cpp"), "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return C.CDLL(so)


def _truth():
    """The reference's own functions when they were compiled here, the oracle's restatement (bit-equal to them, tests/test_oracle_bsdf.py) otherwise."""
    return O.microfacet("ref" if os.path.exists(O.MFREF_SO) else "port")


def _dirs(rng, n, upper):
    d = rng.normal(size=(n, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    if upper:
        d[:, 2] = np.abs(d[:, 2])
    return np.ascontiguousarray(d, np.float32)


@pytest.mark.parametrize("type_", [0, 1])
@pytest.mark.parametrize("alpha", [0.01, 0.1, 0.6])
def test_device_microfacet_source_equals_the_reference(dev, type_, alpha):
    ref = _truth(); rng = np.random.default_rng(7 + 10 * type_ + int(100 * alpha)); n = 100000
    m, v, wi = _dirs(rng, n, False), _dirs(rng, n, False), _dirs(rng, n, True)
    wi[:500] = [0, 0, 1]; wi[500:1000, 2] = 1e-3 * rng.random(500); wi[500:1000] /= np.linalg.norm(wi[500:1000], axis=1, keepdims=True)
    smp = rng.random((n, 2), dtype=np.float32)
    out = np.zeros(n, np.float32)
    dev.dev_mf_eval.argtypes = [C.c_int, C.c_float, C.c_size_t, f32p, f32p]
    dev.dev_mf_eval(type_, alpha, n, m.ctypes.data_as(f32p), out.ctypes.data_as(f32p)); assert np.array_equal(out, ref.eval(type_, alpha, m))
    dev.dev_mf_smith_g1.argtypes = [C.c_int, C.c_float, C.c_size_t, f32p, f32p, f32p]
    dev.dev_mf_smith_g1(type_, alpha, n, v.ctypes.data_as(f32p), m.ctypes.data_as(f32p), out.ctypes.data_as(f32p)); assert np.array_equal(out, ref.smith_g1(type_, alpha, v, m))
    ma = np.ascontiguousarray(np.abs(m))
    dev.dev_mf_pdf.argtypes = [C.c_int, C.c_float, C.c_size_t, f32p, f32p, f32p]
    dev.dev_mf_pdf(type_, alpha, n, wi.ctypes.data_as(f32p), ma.ctypes.data_as(f32p), out.ctypes.data_as(f32p)); assert np.array_equal(out, ref.pdf(type_, alpha, wi, ma))
    mo = np.zeros((n, 3), np.float32); po = np.zeros(n, np.float32)
    dev.dev_mf_sample.argtypes = [C.c_int, C.c_float, C.c_size_t, f32p, f32p, f32p, f32p]
    dev.dev_mf_sample(type_, alpha, n, wi.ctypes.data_as(f32p), smp.ctypes.data_as(f32p), mo.ctypes.data_as(f32p), po.ctypes.data_as(f32p))
    mr, pr = ref.sample(type_, alpha, wi, smp)
    ok = np.isfinite(mr).all(axis=1)
    assert ok.mean() > 0.999 and np.array_equal(mo[ok], mr[ok]) and np.array_equal(po[ok], pr[ok])


def test_device_helper_sources_equal_the_reference(dev):
    ref = _truth(); rng = np.random.default_rng(3); n = 100000
    x = np.concatenate([rng.uniform(-0.999999, 0.999999, n), rng.uniform(-6, 6, 1000)]).astype(np.float32)
    a = np.zeros_like(x); b = np.zeros_like(x)
    dev.dev_erf.argtypes = [C.c_size_t, f32p, f32p, f32p]
    dev.dev_erf(len(x), x.ctypes.data_as(f32p), a.ctypes.data_as(f32p), b.ctypes.data_as(f32p))
    er, eir = ref.erf(x)
    assert np.array_equal(a, er) and np.array_equal(b[np.abs(x) < 1], eir[np.abs(x) < 1])
    c = np.concatenate([rng.uniform(-1, 1, n), [0.0, 1.0, -1.0, 1e-6]]).astype(np.float32)
    f = np.zeros_like(c); ct = np.zeros_like(c)
    dev.dev_fresnel_dielectric_ext.argtypes = [C.c_size_t, f32p, C.c_float, f32p, f32p]
    for eta in (1.0, 1.5046 / 1.000277, 1 / 1.5, 1.33):
        dev.dev_fresnel_dielectric_ext(len(c), c.ctypes.data_as(f32p), eta, f.ctypes.data_as(f32p), ct.ctypes.data_as(f32p))
        fr, tr = ref.fresnel_dielectric_ext(c, eta)
        assert np.array_equal(f, fr) and np.array_equal(ct, tr)
    ca = np.ascontiguousarray(np.abs(c)); out3 = np.zeros((len(c), 3), np.float32)
    dev.dev_fresnel_conductor_exact.argtypes = [C.c_size_t, f32p, f32p, f32p, f32p]
    for eta, k in (((0.2, 0.9, 1.1), (3.9, 2.4, 2.2)), ((1.65746, 0.880369, 0.521229), (9.22387, 6.26952, 4.837)), ((0, 0, 0), (1, 1, 1))):
        e = np.float32(eta); kk = np.float32(k)
        dev.dev_fresnel_conductor_exact(len(c), ca.ctypes.data_as(f32p), e.ctypes.data_as(f32p), kk.ctypes.data_as(f32p), out3.ctypes.data_as(f32p))
        assert np.array_equal(out3, ref.fresnel_conductor_exact(ca, eta, k))
    d = _dirs(rng, n, False); d[:3] = np.eye(3)
    bo = np.zeros_like(d); co = np.zeros_like(d)
    dev.dev_coordinate_system.argtypes = [C.c_size_t, f32p, f32p, f32p]
    dev.dev_coordinate_system(n, d.ctypes.data_as(f32p), bo.ctypes.data_as(f32p), co.ctypes.data_as(f32p))
    br, cr = ref.coordinate_system(d)
    assert np.array_equal(bo, br) and np.array_equal(co, cr)
    smp = rng.random((n, 2), dtype=np.float32); smp[:3] = [[0.5, 0.5], [0, 0], [0.99999994, 0.5]]
    vo = np.zeros((n, 3), np.float32)
    dev.dev_square_to_cosine_hemisphere.argtypes = [C.c_size_t, f32p, f32p]
    dev.dev_square_to_cosine_hemisphere(n, smp.ctypes.data_as(f32p), vo.ctypes.data_as(f32p))
    assert np.array_equal(vo, ref.square_to_cosine_hemisphere(smp))


def test_device_triangle_test_and_transmittance_sources_equal_the_reference(dev):
    """tri_intersect on the accel rows ppg_set_scene packs, fed with the reference's own TriAccel constants: same hit decision, same (t, u, v) as TriAccel::rayIntersect."""
    truth = C.CDLL(O.MFREF_SO) if os.path.exists(O.MFREF_SO) else O.load("port"); name = "mfref_triaccel" if os.path.exists(O.MFREF_SO) else "ppgo_triaccel"
    rng = np.random.default_rng(5); n = 200000
    A = rng.normal(size=(n, 3)).astype(np.float32) * 10; B = A + rng.normal(size=(n, 3)).astype(np.float32); Cc = A + rng.normal(size=(n, 3)).astype(np.float32)
    B[:100] = A[:100]
    w = rng.random((n, 2)); tgt = A + (B - A) * (w[:, :1] * 1.4 - 0.2) + (Cc - A) * (w[:, 1:] * 1.4 - 0.2)
    o = (tgt + rng.normal(size=(n, 3)) * 5).astype(np.float32); d = tgt - o; d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    mint = np.full(n, 1e-4, np.float32); maxt = np.where(rng.random(n) < 0.1, 3.0, np.inf).astype(np.float32)
    k = np.zeros(n, np.int32); c9 = np.zeros((n, 9), np.float32); hit = np.zeros(n, np.uint8); tuv = np.zeros((n, 3), np.float32)
    fn = getattr(truth, name); fn.argtypes = [C.c_size_t] + [f32p] * 7 + [C.POINTER(C.c_int), f32p, C.POINTER(C.c_ubyte), f32p]
    arrs = [np.ascontiguousarray(a, np.float32) for a in (A, B, Cc, o, d, mint, maxt)]
    fn(n, *[a.ctypes.data_as(f32p) for a in arrs], k.ctypes.data_as(C.POINTER(C.c_int)), c9.ctypes.data_as(f32p), hit.ctypes.data_as(C.POINTER(C.c_ubyte)), tuv.ctypes.data_as(f32p))
    hit2 = np.zeros(n, np.uint8); tuv2 = np.zeros((n, 3), np.float32)
    dev.dev_tri_intersect.argtypes = [C.c_size_t, C.POINTER(C.c_int), f32p, f32p, f32p, f32p, f32p, C.POINTER(C.c_ubyte), f32p]
    dev.dev_tri_intersect(n, k.ctypes.data_as(C.POINTER(C.c_int)), c9.ctypes.data_as(f32p), arrs[3].ctypes.data_as(f32p), arrs[4].ctypes.data_as(f32p), mint.ctypes.data_as(f32p),
                          maxt.ctypes.data_as(f32p), hit2.ctypes.data_as(C.POINTER(C.c_ubyte)), tuv2.ctypes.data_as(f32p))
    assert 0.1 < hit.mean() < 0.5 and np.array_equal(hit, hit2) and np.array_equal(tuv[hit == 1], tuv2[hit == 1])
    from ppg_b200 import rtrans
    lut, _ = rtrans.reduce_for_material("beckmann", 1.49, 0.1); lut = np.ascontiguousarray(lut, np.float32)
    cs = np.concatenate([rng.uniform(-0.2, 1, 100000), [0.0, 1.0]]).astype(np.float32)
    a = np.zeros_like(cs); b = np.zeros_like(cs)
    dev.dev_rough_transmittance.argtypes = [C.c_size_t, f32p, f32p, f32p]
    dev.dev_rough_transmittance(len(cs), cs.ctypes.data_as(f32p), lut.ctypes.data_as(f32p), a.ctypes.data_as(f32p))
    port = O.load("port"); port.ppgo_rough_transmittance.argtypes = [C.c_size_t, f32p, f32p, f32p]
    port.ppgo_rough_transmittance(len(cs), cs.ctypes.data_as(f32p), lut.ctypes.data_as(f32p), b.ctypes.data_as(f32p))
    assert np.array_equal(a, b)                                                     # (the oracle's lookup is itself checked against evalCubicInterp1D, tests/test_oracle_bsdf.py)


def _material(name):
    """One BSDF configuration of the hot path (DESIGN.md 1.1) with the wrappers that change its arithmetic: (ppg_bsdf, tables).  Built inside the test: the
    rough-plastic tables are reduced from the nodes of Mitsuba's data files stored under tests/golden."""
    from ppg_b200 import scene as S
    mk = lambda **kw: O.make_bsdf(**kw)
    if name in ROUGHPLASTICS:
        tables = []
        row = S.make_roughplastic(*ROUGHPLASTICS[name], tables)
        return O.bsdf_from_row(row), np.ascontiguousarray(tables, np.float32)
    if name == "plastic nonlinear":
        return O.bsdf_from_row(S.make_plastic(0, (0.6, 0.3, 0.2), (1, 1, 1), 1.49, True)), None
    if name == "plastic twosided":
        return O.bsdf_from_row(S.make_plastic(1, (0.2, 0.3, 0.6), (0.8, 0.8, 0.8), 1.9, False)), None
    if name.startswith("mask"):
        m = mk(type=0, flags=1 | 4, reflectance=(0.6, 0.5, 0.4)) if "diffuse" in name else mk(type=4, flags=4, reflectance=(1, 1, 1), eta=(0.2, 0.9, 1.1), k=(3.9, 2.4, 2.2), alpha=0.2, distribution=1)
        op = (0.6, 0.5, 0.7) if "diffuse" in name else (0.3, 0.3, 0.3)
        m.opacity[0], m.opacity[1], m.opacity[2] = op
        return m, None
    return mk(**SIMPLE[name]), None


SIMPLE = {
    "diffuse": dict(type=0, reflectance=(0.6, 0.5, 0.4)),
    "diffuse twosided": dict(type=0, flags=1, reflectance=(0.6, 0.5, 0.4)),
    "black (emitter without a BSDF)": dict(type=1, reflectance=(0, 0, 0)),                 # (the loaders hand NULL_BLACK over with zero reflectance)
    "dielectric bk7": dict(type=2, reflectance=(1, 1, 1), transmittance=(1, 1, 1), eta=(1.5046 / 1.000277,) * 3),
    "conductor": dict(type=3, reflectance=(1, 1, 1), eta=(0.2, 0.9, 1.1), k=(3.9, 2.4, 2.2)),
    "roughconductor ggx 0.1 twosided": dict(type=4, flags=1, reflectance=(1, 1, 1), eta=(1.65746, 0.880369, 0.521229), k=(9.22387, 6.26952, 4.837), alpha=0.1, distribution=1),
    "roughconductor beckmann 0.3": dict(type=4, reflectance=(0.9, 0.9, 0.9), eta=(0.2, 0.9, 1.1), k=(3.9, 2.4, 2.2), alpha=0.3, distribution=0),
    "roughdielectric ggx 0.1": dict(type=6, reflectance=(1, 1, 1), transmittance=(1, 1, 1), eta=(1.5,) * 3, alpha=0.1, distribution=1),
    "roughdielectric beckmann 0.3 tinted": dict(type=6, reflectance=(0.9, 0.8, 1), transmittance=(0.7, 0.9, 1), eta=(1.33,) * 3, alpha=0.3, distribution=0),
    "thindielectric": dict(type=8, reflectance=(1, 1, 1), transmittance=(0.9, 0.95, 1), eta=(1.5,) * 3),
}
ROUGHPLASTICS = {"roughplastic ggx 0.2": (0, (0.256, 0.013, 0.08), (1, 1, 1), 1.5 / 1.000277, 0.2, 1, False),
                 "roughplastic beckmann 0.4 nonlinear twosided": (1, (0.5, 0.4, 0.3), (0.9, 0.9, 0.9), 1.49, 0.4, 0, True)}
MATERIALS = list(SIMPLE) + list(ROUGHPLASTICS) + ["plastic nonlinear", "plastic twosided", "mask over twosided diffuse", "mask over roughconductor"]


@pytest.mark.parametrize("name", MATERIALS)
def test_device_bsdf_sources_equal_the_oracle(dev, name):
    """bsdf_eval / bsdf_pdf / bsdf_sample of csrc/ppg_device.cuh (host-compiled) against the oracle's restatement of the same Mitsuba models, on the same directions and
    random numbers: every value bit for bit -- eval and pdf on 10^5 direction pairs over the whole sphere (both sides of the surface), sampling on 10^5 (wi, u) pairs
    incl. the model's own extra draw (roughdielectric) and the delta / null lobes."""
    b, tables = _material(name)
    rng = np.random.default_rng(MATERIALS.index(name)); n = 100000
    wi, wo = _dirs(rng, n, False), _dirs(rng, n, False)
    wi[:200, 2] = np.abs(wi[:200, 2]) * 1e-3; wi[:200] /= np.linalg.norm(wi[:200], axis=1, keepdims=True)         # grazing incidence
    wo[200:1200] = wi[200:1200] * [-1, -1, 1]                                                                    # the mirror direction (delta lobes evaluate to 0 without the discrete measure)
    tp = tables.ctypes.data_as(f32p) if tables is not None else None
    ev = np.zeros((n, 3), np.float32); pd = np.zeros(n, np.float32)
    dev.dev_bsdf_eval_pdf.argtypes = [C.POINTER(type(b)), C.c_size_t, f32p, f32p, f32p, f32p, f32p]
    dev.dev_bsdf_eval_pdf(C.byref(b), n, wi.ctypes.data_as(f32p), wo.ctypes.data_as(f32p), ev.ctypes.data_as(f32p), pd.ctypes.data_as(f32p), tp)
    ev0, pd0 = O.bsdf_eval_pdf(b, wi, wo, tables=tables)
    assert np.array_equal(ev.view(np.uint32), ev0.view(np.uint32)) and np.array_equal(pd.view(np.uint32), pd0.view(np.uint32))
    smp = rng.random((n, 2), dtype=np.float32)
    so = np.zeros((n, 3), np.float32); sw = np.zeros((n, 3), np.float32); sp = np.zeros(n, np.float32); sd = np.zeros(n, np.uint8)
    dev.dev_bsdf_sample.argtypes = [C.POINTER(type(b)), C.c_size_t, f32p, f32p, f32p, f32p, f32p, C.POINTER(C.c_ubyte), f32p]
    dev.dev_bsdf_sample(C.byref(b), n, wi.ctypes.data_as(f32p), smp.ctypes.data_as(f32p), so.ctypes.data_as(f32p), sw.ctypes.data_as(f32p), sp.ctypes.data_as(f32p), sd.ctypes.data_as(C.POINTER(C.c_ubyte)), tp)
    so0, sw0, sp0, sd0 = O.bsdf_sample(b, wi, smp, tables=tables)
    lit = (sw0 != 0).any(axis=1)                                                    # a failed sample carries weight 0; its wo is unspecified on both sides
    assert np.array_equal(lit, (sw != 0).any(axis=1)) and (lit.mean() > 0.2 or b.type == 1)
    assert np.array_equal(sw[lit].view(np.uint32), sw0[lit].view(np.uint32)) and np.array_equal(so[lit].view(np.uint32), so0[lit].view(np.uint32))
    assert np.array_equal(sp[lit].view(np.uint32), sp0[lit].view(np.uint32)) and np.array_equal(sd[lit], sd0[lit])


def test_device_texture_source_equals_the_oracle(dev):
    """tex_eval (BitmapTexture::eval -> TMIPMap::evalBilinear, level 0) and tex_gradient_lum (evalGradientBilinear -> the luminances BumpMap::getFrame uses) of the
    device source on the textures of the cbox-textured fixture (RGB and one-channel, repeat / clamp / mirror wrapping, uv scale and offset), packed the way
    ppg_set_scene packs them, against the oracle's texture code at 10^5 texture coordinates reaching far outside [0, 1]^2: bit for bit."""
    from common import load_fixture_scene
    from ppg_b200 import capi
    sc = load_fixture_scene("cbox-textured")
    o = O.Oracle(O.params_from_xml(sc.integrator), sc, kind="port")
    lib = O.load("port"); lib.ppgo_texture_eval.argtypes = [C.c_void_p, C.c_uint32, C.c_size_t, f32p, f32p, f32p]
    arrays = o.scene_arrays
    rng = np.random.default_rng(17); n = 100000
    uv = (rng.random((n, 2)) * 6 - 2.5).astype(np.float32); uv[:4] = [[0, 0], [1, 1], [0.5, 0.5], [np.nan, 0.3]]
    dev.dev_texture_eval.argtypes = [C.POINTER(capi.PpgTexture), C.POINTER(C.c_uint16), C.c_size_t, f32p, f32p, f32p]
    assert len(sc.textures) == 3
    for k in range(len(sc.textures)):
        a = np.zeros((n, 3), np.float32); ga = np.zeros((n, 2), np.float32); b = np.zeros((n, 3), np.float32); gb = np.zeros((n, 2), np.float32)
        assert lib.ppgo_texture_eval(o.h, k, n, uv.ctypes.data_as(f32p), a.ctypes.data_as(f32p), ga.ctypes.data_as(f32p)) == 0
        t = capi.PpgTexture.from_buffer_copy(np.ascontiguousarray(sc.textures[k:k + 1]).tobytes())
        texels = np.ascontiguousarray(sc.texels, np.uint16)
        dev.dev_texture_eval(C.byref(t), texels.ctypes.data_as(C.POINTER(C.c_uint16)), n, uv.ctypes.data_as(f32p), b.ctypes.data_as(f32p), gb.ctypes.data_as(f32p))
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and np.array_equal(ga.view(np.uint32), gb.view(np.uint32)), k
        assert np.abs(a[4:]).max() > 0.1 and np.abs(ga[4:]).max() > 0


def test_device_discrete_sampling_source_equals_the_reference(dev):
    """cdf_sample + the sample reuse of the device's sample_emitter_direct on the normalised table ppg_set_scene uploads, against DiscreteDistribution::sampleReuse of the
    reference compiled verbatim (or the oracle's, bit-equal to it): index and reused sample bit for bit, zero-weight entries skipped the same way."""
    have_ref = os.path.exists(O.MFREF_SO)
    truth = C.CDLL(O.MFREF_SO) if have_ref else O.load("port"); name = "mfref_discrete" if have_ref else "ppgo_discrete"
    u32p = C.POINTER(C.c_uint32)
    rng = np.random.default_rng(44)
    for ne in (1, 3, 40, 1000):
        w = rng.lognormal(0, 2, ne).astype(np.float32)
        if ne > 2:
            w[rng.integers(0, ne, max(1, ne // 5))] = 0; w[0] = 0; w[-1] = 0
            w[ne // 2] = max(w[ne // 2], 1e-3)
        n = 100000
        smp = rng.random(n, dtype=np.float32); smp[0] = 0.0
        pdf = np.zeros(ne, np.float32); s = C.c_float(); idx = np.zeros(n, np.uint32); reuse = np.zeros(n, np.float32)
        fn = getattr(truth, name); fn.argtypes = [C.c_size_t, f32p, C.c_size_t, f32p, f32p, C.POINTER(C.c_float), u32p, f32p]
        fn(ne, w.ctypes.data_as(f32p), n, smp.ctypes.data_as(f32p), pdf.ctypes.data_as(f32p), C.byref(s), idx.ctypes.data_as(u32p), reuse.ctypes.data_as(f32p))
        # the table as the host builds it (ppg_host.cu, emitter tables: cumulative sum, x 1/sum, last entry = 1): DiscreteDistribution::normalize
        cdf = np.zeros(ne + 1, np.float32)
        for i in range(ne):
            cdf[i + 1] = np.float32(cdf[i] + w[i])
        nrm = np.float32(1.0) / cdf[-1]; cdf[1:] = cdf[1:] * nrm; cdf[-1] = 1.0
        assert np.array_equal(np.diff(cdf), pdf) or np.allclose(np.diff(cdf), pdf, rtol=0, atol=0)
        idx2 = np.zeros(n, np.uint32); reuse2 = np.zeros(n, np.float32)
        dev.dev_discrete.argtypes = [C.c_size_t, f32p, C.c_size_t, f32p, u32p, f32p]
        dev.dev_discrete(ne, cdf.ctypes.data_as(f32p), n, smp.ctypes.data_as(f32p), idx2.ctypes.data_as(u32p), reuse2.ctypes.data_as(f32p))
        assert np.array_equal(idx, idx2) and np.array_equal(reuse.view(np.uint32), reuse2.view(np.uint32)), ne


def test_device_sdtree_sources_against_the_reference_trees(dev):
    """stree_lookup (through the prefix table stree_table_kernel builds -- the __global__ function runs here as a plain loop), dtree_pdf, dtree_sample and the
    cylindrical maps of the device source on trees trained by the oracle (the reference's own SD-tree code where oracle/_ref exists): leaf index and voxel size bit
    for bit; sampled directions within 2e-6 (the fold of the per-level origins is the reference's, the two leaf numbers enter in its order); pdf to 2e-6 relative
    (top-down product here, bottom-up recursion there) -- the tolerances of the same comparison on the GPU (tests/test_gpu_parity.py::test_op_*)."""
    from common import load_cbox
    sc = load_cbox(96)
    o = O.Oracle(O.params_from_xml(dict(sc.integrator, budget="60")), sc, kind="ref" if O.have_ref() else "port"); o.render()
    e = o.export(0)
    rng = np.random.default_rng(8); n = 100000
    mn, mx = e["aabb"]; ext = (mx - mn).astype(np.float32)
    pts = (mn + rng.random((n, 3)) * (mx - mn)).astype(np.float32); pts[:8] = [mn, mx, (mn + mx) / 2, mn - 1, mx + 1, [mn[0], mx[1], mn[2]], [mx[0], mn[1], mx[2]], (mn + mx) / 2 + 1e-3]
    leaf, size = o.lookup(pts)
    u32p = C.POINTER(C.c_uint32)
    sch = np.ascontiguousarray(e["s_children"], np.uint32); gl = np.zeros(n, np.uint32); gs = np.zeros((n, 3), np.float32)
    dev.dev_stree_lookup.argtypes = [u32p, C.c_size_t, f32p, f32p, f32p, C.c_size_t, u32p, f32p]
    dev.dev_stree_lookup(sch.ctypes.data_as(u32p), len(sch), np.float32(mn).ctypes.data_as(f32p), ext.ctypes.data_as(f32p), pts.ctypes.data_as(f32p), n, gl.ctypes.data_as(u32p), gs.ctypes.data_as(f32p))
    assert np.array_equal(gl, leaf) and np.array_equal(gs, size) and len(np.unique(leaf)) > 10
    leaves = np.nonzero(e["s_is_leaf"])[0].astype(np.uint32)
    ql = rng.choice(leaves, n).astype(np.uint32)
    d = rng.normal(size=(n, 3)).astype(np.float32); d /= np.linalg.norm(d, axis=1, keepdims=True)
    rnd = rng.random((n, 24), dtype=np.float32)
    pdf = np.zeros(n, np.float32); dirs = np.zeros((n, 3), np.float32)
    sums = np.ascontiguousarray(e["sums"], np.float32); ch = np.ascontiguousarray(e["children"], np.uint16); first = e["tree_first"].astype(np.uint32)
    dev.dev_dtree.argtypes = [f32p, C.POINTER(C.c_uint16), C.c_size_t, u32p, f32p, f32p, u32p, f32p, f32p, C.c_size_t, C.c_size_t, f32p, f32p]
    dev.dev_dtree(sums.ctypes.data_as(f32p), ch.ctypes.data_as(C.POINTER(C.c_uint16)), len(sums), first.ctypes.data_as(u32p), e["tree_sum"].ctypes.data_as(f32p),
                  e["tree_weight"].ctypes.data_as(f32p), ql.ctypes.data_as(u32p), d.ctypes.data_as(f32p), rnd.ctypes.data_as(f32p), 24, n, pdf.ctypes.data_as(f32p), dirs.ctypes.data_as(f32p))
    ref_pdf = o.pdf(ql, d); ref_dir = o.sample(ql, rnd)
    assert np.allclose(pdf, ref_pdf, rtol=2e-6, atol=1e-12) and np.abs(dirs - ref_dir).max() <= 2e-6
    assert (dirs == ref_dir).all(axis=1).mean() > 0.9                              # (mostly bit-equal: same libm here)
