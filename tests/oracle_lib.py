"""Test-side ctypes wrapper of the CPU oracle (oracle/libppg_oracle.so and, when it was
built, oracle/_ref/libppg_oracle_ref.so = same tracer on the reference's verbatim SD-tree).
Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import this."""
import ctypes as C
import os
import subprocess

import numpy as np

from ppg_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PORT_SO = os.path.join(ROOT, "oracle", "libppg_oracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libppg_oracle_ref.so")


def build():
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle")], check=True)


def _declare(lib):
    H = C.c_void_p
    f32p = C.POINTER(C.c_float); u32p = C.POINTER(C.c_uint32); u8p = C.POINTER(C.c_uint8); u16p = C.POINTER(C.c_uint16)
    i32p = C.POINTER(C.c_int32); u64p = C.POINTER(C.c_uint64)
    lib.ppgo_create.restype = H
    lib.ppgo_create.argtypes = [C.POINTER(capi.PpgParams), C.POINTER(capi.PpgSceneDesc), f32p, f32p, C.c_int]
    lib.ppgo_destroy.argtypes = [H]; lib.ppgo_destroy.restype = None
    lib.ppgo_render.argtypes = [H, f32p, C.POINTER(capi.PpgStats)]
    lib.ppgo_set_capture.argtypes = [H, f32p, i32p]
    lib.ppgo_set_shard.argtypes = [H, C.c_int, C.c_int]
    lib.ppgo_set_allreduce.argtypes = [H, capi.ALLREDUCE_FN, C.c_void_p]
    lib.ppgo_step_reset.argtypes = [H, C.c_int]
    lib.ppgo_step_passes.argtypes = [H, C.c_int, C.c_int, f32p]
    lib.ppgo_step_build.argtypes = [H, C.POINTER(capi.PpgIterationStats)]
    lib.ppgo_get_moment_images.argtypes = [H, f32p, f32p]
    lib.ppgo_bsdf_eval_pdf.argtypes = [C.POINTER(capi.PpgBsdf), C.c_size_t, f32p, f32p, f32p, f32p, f32p]
    lib.ppgo_bsdf_sample.argtypes = [C.POINTER(capi.PpgBsdf), C.c_size_t, f32p, f32p, f32p, f32p, f32p, u8p, f32p]
    for fn, at in (("eval", [C.c_int, C.c_float, C.c_size_t, f32p, f32p]), ("smith_g1", [C.c_int, C.c_float, C.c_size_t, f32p, f32p, f32p]),
                   ("pdf", [C.c_int, C.c_float, C.c_size_t, f32p, f32p, f32p]), ("sample", [C.c_int, C.c_float, C.c_size_t, f32p, f32p, f32p, f32p])):
        getattr(lib, "ppgo_mf_" + fn).argtypes = at
    lib.ppgo_mf_erf.argtypes = [C.c_size_t, f32p, f32p, f32p]
    lib.ppgo_emitter_sample_direct.argtypes = [H, C.c_size_t, f32p, f32p, f32p, C.c_int, f32p, f32p, f32p, f32p]
    lib.ppgo_env_pdf.argtypes = [H, C.c_size_t, f32p, f32p, f32p]
    lib.ppgo_tree_dump.argtypes = [H, C.c_char_p, f32p]
    lib.ppgo_tree_commit.argtypes = [H, C.c_size_t] + [f32p] * 9 + [u8p, f32p, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.ppgo_tree_refine.argtypes = [H, C.c_uint64, C.c_int]
    lib.ppgo_tree_reset.argtypes = [H, C.c_int, C.c_float]
    lib.ppgo_tree_build.argtypes = [H]
    lib.ppgo_tree_record.argtypes = [H, C.c_size_t, f32p, f32p, f32p, f32p, f32p, f32p, f32p, f32p, u8p, f32p, C.c_int, C.c_int, C.c_int]
    lib.ppgo_tree_lookup.argtypes = [H, C.c_size_t, f32p, u32p, f32p]
    lib.ppgo_tree_pdf.argtypes = [H, C.c_size_t, u32p, f32p, f32p]
    lib.ppgo_tree_sample.argtypes = [H, C.c_size_t, u32p, f32p, C.c_size_t, f32p]
    lib.ppgo_tree_fraction.argtypes = [H, C.c_size_t, u32p, f32p]
    lib.ppgo_tree_counts.argtypes = [H, u64p]
    if hasattr(lib, "ppgo_tree_set_adam"):          # (a reference oracle built before this entry point existed lacks it)
        lib.ppgo_tree_set_adam.argtypes = [H, C.c_uint32, f32p]
    lib.ppgo_tree_export.argtypes = [H, C.c_int, u32p, i32p, u8p, u64p, u32p, f32p, f32p, i32p, f32p, u16p, f32p, f32p]
    return lib


_libs = {}


def load(kind="port"):
    if kind not in _libs:
        path = PORT_SO if kind == "port" else REF_SO
        if not os.path.exists(path):
            if kind == "port":
                build()
            else:
                raise FileNotFoundError(path)
        _libs[kind] = _declare(C.CDLL(path))
    return _libs[kind]


def have_ref():
    return os.path.exists(REF_SO)


def default_params(**kw):
    """Reference defaults (GP:1014-1085, integrator.cpp:190-225), restated on the test side."""
    p = capi.PpgParams()
    p.nee = 0; p.sample_combination = 1; p.spatial_filter = 0; p.directional_filter = 0; p.bsdf_sampling_fraction_loss = 0
    p.sd_tree_max_memory = -1; p.s_tree_threshold = 12000; p.d_tree_threshold = 0.01; p.bsdf_sampling_fraction = 0.5
    p.spp_per_pass = 4; p.budget_type = 1; p.budget = 300.0; p.dump_sd_tree = 0
    p.max_depth = -1; p.rr_depth = 5; p.strict_normals = 0; p.hide_emitters = 0; p.seed = 1234
    for k, v in kw.items():
        setattr(p, k, v)
    return p


_ENUMS = {
    "nee": {"never": 0, "kickstart": 1, "always": 2},
    "sampleCombination": {"discard": 0, "automatic": 1, "inversevar": 2},
    "spatialFilter": {"nearest": 0, "stochastic": 1, "box": 2},
    "directionalFilter": {"nearest": 0, "box": 1},
    "bsdfSamplingFractionLoss": {"none": 0, "kl": 1, "var": 2},
    "budgetType": {"spp": 0, "seconds": 1},
}
_FIELDS = {
    "nee": "nee", "sampleCombination": "sample_combination", "spatialFilter": "spatial_filter",
    "directionalFilter": "directional_filter", "bsdfSamplingFractionLoss": "bsdf_sampling_fraction_loss",
    "sdTreeMaxMemory": "sd_tree_max_memory", "sTreeThreshold": "s_tree_threshold", "dTreeThreshold": "d_tree_threshold",
    "bsdfSamplingFraction": "bsdf_sampling_fraction", "sppPerPass": "spp_per_pass", "budgetType": "budget_type",
    "budget": "budget", "dumpSDTree": "dump_sd_tree", "maxDepth": "max_depth", "rrDepth": "rr_depth",
    "strictNormals": "strict_normals", "hideEmitters": "hide_emitters", "seed": "seed",
}


def params_from_xml(props: dict, **override):
    """XML (name -> string) to ppg_params, on the test side (the product does this in C: ppg_params_set)."""
    p = default_params()
    allp = dict(props); allp.update({k: str(v) for k, v in override.items()})
    for k, v in allp.items():
        f = _FIELDS[k]
        if k in _ENUMS:
            setattr(p, f, _ENUMS[k][v])
        elif v in ("true", "false"):
            setattr(p, f, 1 if v == "true" else 0)
        elif f in ("d_tree_threshold", "bsdf_sampling_fraction", "budget"):
            setattr(p, f, float(v))
        else:
            setattr(p, f, int(float(v)))
    return p


def fptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


class Oracle:
    def __init__(self, params, scene=None, aabb=None, nthreads=0, kind="port"):
        self.lib = load(kind)
        self.kind = kind
        self.scene_arrays = capi.SceneArrays(scene) if scene is not None else None
        self.params = params
        if scene is not None:
            self.W, self.H = scene.film_width, scene.film_height
            self.h = self.lib.ppgo_create(C.byref(params), C.byref(self.scene_arrays.desc), None, None, nthreads)
        else:
            mn = np.asarray(aabb[0], np.float32); mx = np.asarray(aabb[1], np.float32)
            self.h = self.lib.ppgo_create(C.byref(params), None, fptr(mn), fptr(mx), nthreads)

    def close(self):
        if self.h:
            self.lib.ppgo_destroy(self.h); self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_shard(self, rank, world):
        assert self.lib.ppgo_set_shard(self.h, rank, world) == 0

    def set_allreduce(self, fn):
        """fn(numpy float32 view) sums in place over ranks (host memory)."""
        def _cb(user, ptr, n):
            a = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_float)), shape=(n,))
            fn(a)
            return 0
        self._cb = capi.ALLREDUCE_FN(_cb)
        assert self.lib.ppgo_set_allreduce(self.h, self._cb, None) == 0

    def render(self, capture=False):
        img = np.zeros((self.H, self.W, 3), np.float32)
        st = capi.PpgStats()
        cap = None
        if capture:
            n = self.W * self.H * self.params.spp_per_pass
            self._capli = np.zeros((n, 3), np.float32); self._capd = np.zeros(n, np.int32)
            self.lib.ppgo_set_capture(self.h, fptr(self._capli), self._capd.ctypes.data_as(C.POINTER(C.c_int32)))
            cap = (self._capli, self._capd)
        rc = self.lib.ppgo_render(self.h, fptr(img), C.byref(st))
        assert rc == 0, rc
        return (img, st.as_dict(), cap) if capture else (img, st.as_dict())

    # ---- step-wise
    def set_capture(self):
        n = self.W * self.H * self.params.spp_per_pass
        self._capli = np.zeros((n, 3), np.float32); self._capd = np.zeros(n, np.int32)
        self.lib.ppgo_set_capture(self.h, fptr(self._capli), self._capd.ctypes.data_as(C.POINTER(C.c_int32)))
        return self._capli, self._capd

    def step_reset(self, it):
        assert self.lib.ppgo_step_reset(self.h, it) == 0

    def step_passes(self, n, is_final=False):
        v = C.c_float(0)
        assert self.lib.ppgo_step_passes(self.h, n, int(is_final), C.byref(v)) == 0
        return v.value

    def step_build(self):
        st = capi.PpgIterationStats()
        assert self.lib.ppgo_step_build(self.h, C.byref(st)) == 0
        return st.as_dict()

    def moment_images(self):
        a = np.zeros((self.H, self.W, 4), np.float32); b = np.zeros_like(a)
        self.lib.ppgo_get_moment_images(self.h, fptr(a), fptr(b))
        return a, b

    # ---- tree level
    def emitter_sample_direct(self, ref, ref_n, smp, max_interactions=-1):
        """Scene::sampleAttenuatedEmitterDirect at the points `ref`: (d, value, pdf, dist); pdf == 0 where the sample carries nothing."""
        ref = np.ascontiguousarray(ref, np.float32); ref_n = np.ascontiguousarray(ref_n, np.float32); smp = np.ascontiguousarray(smp, np.float32)
        n = len(ref); d = np.zeros((n, 3), np.float32); val = np.zeros((n, 3), np.float32); pdf = np.zeros(n, np.float32); dist = np.zeros(n, np.float32)
        rc = self.lib.ppgo_emitter_sample_direct(self.h, n, fptr(ref), fptr(ref_n), fptr(smp), max_interactions, fptr(d), fptr(val), fptr(pdf), fptr(dist))
        assert rc == 0, rc
        return d, val, pdf, dist

    def env_pdf(self, d):
        """(light-sampling density incl. the emitter choice, radiance) of the environment emitter for world directions `d`."""
        d = np.ascontiguousarray(d, np.float32); pdf = np.zeros(len(d), np.float32); val = np.zeros((len(d), 3), np.float32)
        rc = self.lib.ppgo_env_pdf(self.h, len(d), fptr(d), fptr(pdf), fptr(val))
        assert rc == 0, rc
        return pdf, val

    def commit(self, o, d, throughput, bsdf_val, radiance, wo_pdf, bsdf_pdf, dtree_pdf, weight, is_delta, rnd, sfilter=0, dfilter=0, loss=0, verbatim=False):
        """Vertex::commit for n vertices: the restated commit_vertex, or (verbatim, reference backend only) the reference's own struct Vertex."""
        A = lambda a: np.ascontiguousarray(a, np.float32)
        o, d, thr, bv, rad, wp, bp, dp, w, rnd = map(A, (o, d, throughput, bsdf_val, radiance, wo_pdf, bsdf_pdf, dtree_pdf, weight, rnd))
        dl = np.ascontiguousarray(is_delta, np.uint8)
        return self.lib.ppgo_tree_commit(self.h, len(wp), fptr(o), fptr(d), fptr(thr), fptr(bv), fptr(rad), fptr(wp), fptr(bp), fptr(dp), fptr(w),
                                         dl.ctypes.data_as(C.POINTER(C.c_uint8)), fptr(rnd), sfilter, dfilter, loss, 1 if verbatim else 0)

    def dump(self, path, cam_to_world):
        """The .sdt file of the tree's current state, written by the reference's own code (reference backend only)."""
        cam = np.ascontiguousarray(cam_to_world, np.float32).reshape(16)
        return self.lib.ppgo_tree_dump(self.h, str(path).encode(), fptr(cam))

    def refine(self, threshold, max_mb=-1):
        self.lib.ppgo_tree_refine(self.h, int(threshold), max_mb)

    def reset(self, max_depth=20, threshold=0.01):
        self.lib.ppgo_tree_reset(self.h, max_depth, threshold)

    def build(self):
        self.lib.ppgo_tree_build(self.h)

    def record(self, o, d, radiance, wo_pdf, product=None, bsdf_pdf=None, dtree_pdf=None, weight=None, is_delta=None, rnd=None,
               sfilter=0, dfilter=0, loss=0):
        n = len(radiance)
        c = lambda a: None if a is None else fptr(np.ascontiguousarray(a, np.float32))
        keep = [np.ascontiguousarray(x, np.float32) if x is not None else None for x in (o, d, radiance, product, wo_pdf, bsdf_pdf, dtree_pdf, weight, rnd)]
        ptrs = [None if k is None else fptr(k) for k in keep]
        dl = None
        if is_delta is not None:
            dl = np.ascontiguousarray(is_delta, np.uint8)
        self.lib.ppgo_tree_record(self.h, n, ptrs[0], ptrs[1], ptrs[2], ptrs[3], ptrs[4], ptrs[5], ptrs[6], ptrs[7],
                                  None if dl is None else dl.ctypes.data_as(C.POINTER(C.c_uint8)), ptrs[8], sfilter, dfilter, loss)

    def lookup(self, p):
        p = np.ascontiguousarray(p, np.float32); n = len(p)
        leaf = np.zeros(n, np.uint32); size = np.zeros((n, 3), np.float32)
        self.lib.ppgo_tree_lookup(self.h, n, fptr(p), leaf.ctypes.data_as(C.POINTER(C.c_uint32)), fptr(size))
        return leaf, size

    def pdf(self, leaf, d):
        leaf = np.ascontiguousarray(leaf, np.uint32); d = np.ascontiguousarray(d, np.float32)
        out = np.zeros(len(leaf), np.float32)
        self.lib.ppgo_tree_pdf(self.h, len(leaf), leaf.ctypes.data_as(C.POINTER(C.c_uint32)), fptr(d), fptr(out))
        return out

    def sample(self, leaf, rnd):
        leaf = np.ascontiguousarray(leaf, np.uint32); rnd = np.ascontiguousarray(rnd, np.float32)
        out = np.zeros((len(leaf), 3), np.float32)
        self.lib.ppgo_tree_sample(self.h, len(leaf), leaf.ctypes.data_as(C.POINTER(C.c_uint32)), fptr(rnd), rnd.shape[1], fptr(out))
        return out

    def set_adam(self, node, state6):
        """Seed the sampling-fraction optimiser of leaf `node` (iter, m, v, variable, batchAcc, batchGrad)."""
        s = np.ascontiguousarray(state6, np.float32)
        assert s.shape == (6,) and self.lib.ppgo_tree_set_adam(self.h, int(node), fptr(s)) == 0

    def fraction(self, leaf):
        leaf = np.ascontiguousarray(leaf, np.uint32); out = np.zeros(len(leaf), np.float32)
        self.lib.ppgo_tree_fraction(self.h, len(leaf), leaf.ctypes.data_as(C.POINTER(C.c_uint32)), fptr(out))
        return out

    def export(self, which=0):
        cnt = (C.c_uint64 * 4)()
        self.lib.ppgo_tree_counts(self.h, cnt)
        N, nq = int(cnt[0]), int(cnt[2 + which])
        e = dict(
            s_children=np.zeros((N, 2), np.uint32), s_axis=np.zeros(N, np.int32), s_is_leaf=np.zeros(N, np.uint8),
            tree_first=np.zeros(N, np.uint64), tree_count=np.zeros(N, np.uint32), tree_sum=np.zeros(N, np.float32),
            tree_weight=np.zeros(N, np.float32), tree_depth=np.zeros(N, np.int32), sums=np.zeros((nq, 4), np.float32),
            children=np.zeros((nq, 4), np.uint16), adam=np.zeros((N, 6), np.float32), aabb=np.zeros((2, 3), np.float32))
        P = lambda a, t: a.ctypes.data_as(C.POINTER(t))
        self.lib.ppgo_tree_export(self.h, which, P(e["s_children"], C.c_uint32), P(e["s_axis"], C.c_int32), P(e["s_is_leaf"], C.c_uint8),
                                  P(e["tree_first"], C.c_uint64), P(e["tree_count"], C.c_uint32), P(e["tree_sum"], C.c_float),
                                  P(e["tree_weight"], C.c_float), P(e["tree_depth"], C.c_int32), P(e["sums"], C.c_float),
                                  P(e["children"], C.c_uint16), P(e["adam"], C.c_float), P(e["aabb"], C.c_float))
        e["n_leaves"] = int(cnt[1])
        return e


def make_bsdf(type=0, flags=0, reflectance=(0.5, 0.5, 0.5), transmittance=(1, 1, 1), eta=(1.5, 1.5, 1.5), k=(0, 0, 0), alpha=0.1, distribution=1):
    b = capi.PpgBsdf()
    b.type = type; b.flags = flags; b.alpha = alpha; b.distribution = distribution
    for i in range(3):
        b.reflectance[i] = reflectance[i]; b.specular_transmittance[i] = transmittance[i]; b.eta[i] = eta[i]; b.k[i] = k[i]
    return b


def bsdf_from_row(row):
    """ppg_bsdf from one row of SceneDesc.bsdfs."""
    b = capi.PpgBsdf()
    raw = np.ascontiguousarray(row, np.float32).tobytes()
    C.memmove(C.byref(b), raw, min(len(raw), C.sizeof(b)))
    return b


def _tab(tables):
    if tables is None:
        return None, None
    t = np.ascontiguousarray(tables, np.float32)
    return t, fptr(t)


def bsdf_eval_pdf(b, wi, wo, kind="port", tables=None):
    lib = load(kind); wi = np.ascontiguousarray(wi, np.float32); wo = np.ascontiguousarray(wo, np.float32)
    ev = np.zeros_like(wi); pdf = np.zeros(len(wi), np.float32)
    keep, tp = _tab(tables)
    lib.ppgo_bsdf_eval_pdf(C.byref(b), len(wi), fptr(wi), fptr(wo), fptr(ev), fptr(pdf), tp)
    return ev, pdf


def bsdf_sample(b, wi, smp, kind="port", tables=None):
    lib = load(kind); wi = np.ascontiguousarray(wi, np.float32); smp = np.ascontiguousarray(smp, np.float32)
    wo = np.zeros_like(wi); w = np.zeros_like(wi); pdf = np.zeros(len(wi), np.float32); d = np.zeros(len(wi), np.uint8)
    keep, tp = _tab(tables)
    lib.ppgo_bsdf_sample(C.byref(b), len(wi), fptr(wi), fptr(smp), fptr(wo), fptr(w), fptr(pdf), d.ctypes.data_as(C.POINTER(C.c_uint8)), tp)
    return wo, w, pdf, d


MFREF_SO = os.path.join(ROOT, "oracle", "_ref", "libmicrofacet_ref.so")


def microfacet(kind):
    """Entry points of a microfacet distribution: kind "port" = the restated struct of the oracle, "ref" = the reference's MicrofacetDistribution
    compiled verbatim (oracle/_ref/libmicrofacet_ref.so).  Returns an object with eval / smith_g1 / pdf / sample / erf over numpy arrays."""
    f32p = C.POINTER(C.c_float)
    if kind == "ref":
        lib = C.CDLL(MFREF_SO); pre = "mfref_"; hp = "mfref_"
        for fn, at in (("eval", [C.c_int, C.c_float, C.c_size_t, f32p, f32p]), ("smith_g1", [C.c_int, C.c_float, C.c_size_t, f32p, f32p, f32p]),
                       ("pdf", [C.c_int, C.c_float, C.c_size_t, f32p, f32p, f32p]), ("sample", [C.c_int, C.c_float, C.c_size_t, f32p, f32p, f32p, f32p])):
            getattr(lib, pre + fn).argtypes = at
        lib.mfref_erf.argtypes = [C.c_size_t, f32p, f32p, f32p]
    else:
        lib = load("port"); pre = "ppgo_mf_"; hp = "ppgo_"

    class MF:
        def eval(self, t, a, m):
            m = np.ascontiguousarray(m, np.float32); out = np.zeros(len(m), np.float32); getattr(lib, pre + "eval")(t, a, len(m), fptr(m), fptr(out)); return out

        def smith_g1(self, t, a, v, m):
            v = np.ascontiguousarray(v, np.float32); m = np.ascontiguousarray(m, np.float32); out = np.zeros(len(m), np.float32)
            getattr(lib, pre + "smith_g1")(t, a, len(m), fptr(v), fptr(m), fptr(out)); return out

        def pdf(self, t, a, wi, m):
            wi = np.ascontiguousarray(wi, np.float32); m = np.ascontiguousarray(m, np.float32); out = np.zeros(len(m), np.float32)
            getattr(lib, pre + "pdf")(t, a, len(m), fptr(wi), fptr(m), fptr(out)); return out

        def sample(self, t, a, wi, smp):
            wi = np.ascontiguousarray(wi, np.float32); smp = np.ascontiguousarray(smp, np.float32); m = np.zeros_like(wi); pdf = np.zeros(len(wi), np.float32)
            getattr(lib, pre + "sample")(t, a, len(wi), fptr(wi), fptr(smp), fptr(m), fptr(pdf)); return m, pdf

        def fresnel_dielectric_ext(self, c, eta):
            c = np.ascontiguousarray(c, np.float32); f = np.zeros_like(c); ct = np.zeros_like(c)
            getattr(lib, hp + "fresnel_dielectric_ext")(C.c_size_t(len(c)), fptr(c), C.c_float(eta), fptr(f), fptr(ct)); return f, ct

        def fresnel_conductor_exact(self, c, eta, k):
            c = np.ascontiguousarray(c, np.float32); e = np.ascontiguousarray(eta, np.float32); kk = np.ascontiguousarray(k, np.float32); out = np.zeros((len(c), 3), np.float32)
            getattr(lib, hp + "fresnel_conductor_exact")(C.c_size_t(len(c)), fptr(c), fptr(e), fptr(kk), fptr(out)); return out

        def coordinate_system(self, a):
            a = np.ascontiguousarray(a, np.float32); b = np.zeros_like(a); c = np.zeros_like(a)
            getattr(lib, hp + "coordinate_system")(C.c_size_t(len(a)), fptr(a), fptr(b), fptr(c)); return b, c

        def square_to_cosine_hemisphere(self, smp):
            smp = np.ascontiguousarray(smp, np.float32); out = np.zeros((len(smp), 3), np.float32)
            getattr(lib, hp + "square_to_cosine_hemisphere")(C.c_size_t(len(smp)), fptr(smp), fptr(out)); return out

        def erf(self, x):
            x = np.ascontiguousarray(x, np.float32); a = np.zeros_like(x); b = np.zeros_like(x); getattr(lib, pre + "erf")(len(x), fptr(x), fptr(a), fptr(b)); return a, b
    return MF()
