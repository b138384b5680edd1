"""Host-side mirror of the reference's integrator plugin surface.

``GuidedPathTracer(props)`` takes the same XML parameter names and string values as
``<integrator type="guided_path">`` (reference: mitsuba/src/integrators/path/guided_path.cpp:1014-1085
plus MonteCarloIntegrator, src/librender/integrator.cpp:190-225), validates them the same way (an unknown
enum string raises, like the reference's ``Assert(false)``) and renders through the C ABI of
libppg_b200.so (include/ppg.h).  All compute happens in the CUDA library; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi
from .scene import SceneDesc


class PpgError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"ppg error {code}: {msg}")
        self.code = code


def _check(lib, rc, allow=()):
    if rc != 0 and rc not in allow:
        raise PpgError(rc, lib.ppg_last_error().decode(errors="replace"))
    return rc


def make_params(props: dict | None = None, **kw) -> capi.PpgParams:
    """Properties -> ppg_params through ppg_params_default / ppg_params_set (values as XML strings)."""
    lib = capi.load_library()
    p = capi.PpgParams()
    lib.ppg_params_default(C.byref(p))
    allp = dict(props or {})
    allp.update(kw)
    for name, value in allp.items():
        if isinstance(value, bool):
            value = "true" if value else "false"
        _check(lib, lib.ppg_params_set(C.byref(p), name.encode(), str(value).encode()))
    _check(lib, lib.ppg_params_validate(C.byref(p)))
    return p


class GuidedPathTracer:
    """CreateInstance(props) + Integrator::render() of the reference plugin, on one B200."""

    description = "Guided path tracer"

    def __init__(self, props: dict | None = None, device: int = -1, **kw):
        self.lib = capi.load_library()
        self.params = make_params(props, **kw)
        self._h = C.c_void_p()
        _check(self.lib, self.lib.ppg_create(C.byref(self.params), device, C.byref(self._h)))
        self._scene_arrays = None
        self._cb = None
        self.W = self.H = 0

    def close(self):
        if self._h:
            self.lib.ppg_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_scene(self, scene: SceneDesc):
        self._scene_arrays = capi.SceneArrays(scene)
        self.W, self.H = scene.film_width, scene.film_height
        _check(self.lib, self.lib.ppg_set_scene(self._h, C.byref(self._scene_arrays.desc)))
        return self

    def set_shard(self, rank: int, world_size: int):
        _check(self.lib, self.lib.ppg_set_shard(self._h, rank, world_size))
        return self

    def set_allreduce(self, fn):
        """fn(device_ptr: int, n_floats: int) -> None must sum the fp32 buffer in place over all ranks."""
        def _cb(user, ptr, n):
            try:
                fn(ptr, n)
                return 0
            except Exception as e:  # noqa: BLE001 - must not propagate through C
                print("allreduce callback failed:", e, flush=True)
                return 1
        self._cb = capi.ALLREDUCE_FN(_cb)
        _check(self.lib, self.lib.ppg_set_allreduce(self._h, self._cb, None))
        return self

    def init_nccl(self, rank: int | None = None, world_size: int | None = None, broadcast=None):
        """Create the library's own NCCL communicator (ppg_nccl_unique_id / ppg_nccl_init): collectives then run on the render stream
        without a host round trip.  The 128-byte unique id of rank 0 reaches the other ranks through `broadcast(bytes_or_None) -> bytes`
        (default: torch.distributed.broadcast_object_list on the default process group -- bootstrap plumbing only)."""
        if broadcast is None:
            import torch.distributed as dist
            rank = dist.get_rank() if rank is None else rank
            world_size = dist.get_world_size() if world_size is None else world_size

            def broadcast(b):
                box = [b]
                dist.broadcast_object_list(box, src=0)
                return box[0]
        buf = C.create_string_buffer(128)
        if rank == 0:
            _check(self.lib, self.lib.ppg_nccl_unique_id(buf))
        ident = broadcast(bytes(buf.raw) if rank == 0 else None)
        buf = C.create_string_buffer(ident, 128)
        _check(self.lib, self.lib.ppg_nccl_init(self._h, buf, rank, world_size))
        return self

    def set_clock(self, fn):
        """budgetType=seconds reads fn() -> seconds since the render started (None: the steady clock)."""
        self._clock = capi.CLOCK_FN(lambda user: float(fn())) if fn is not None else C.cast(None, capi.CLOCK_FN)
        _check(self.lib, self.lib.ppg_set_clock(self._h, self._clock, None))
        return self

    def set_film_callback(self, fn):
        """fn(rgb_device_ptr, width, height, passes_rendered) after every performRenderPasses (progressive film)."""
        self._film = capi.FILM_FN(lambda user, ptr, w, h, n: fn(ptr, w, h, n)) if fn is not None else C.cast(None, capi.FILM_FN)
        _check(self.lib, self.lib.ppg_set_film_callback(self._h, self._film, None))
        return self

    def render(self):
        """Integrator::render(): returns (rgb HxWx3 float32 on the host, stats dict)."""
        img = np.empty((self.H, self.W, 3), np.float32)
        st = capi.PpgStats()
        self.last_status = _check(self.lib, self.lib.ppg_render(self._h, img.ctypes.data_as(C.POINTER(C.c_float)), C.byref(st)), allow=(-5,))   # -5: cancelled, partial film
        return img, st.as_dict()

    def render_device(self):
        """Same, film left in HBM: returns (device pointer of W*H*3 floats, stats dict)."""
        ptr = C.c_void_p()
        st = capi.PpgStats()
        self.last_status = _check(self.lib, self.lib.ppg_render_device(self._h, C.byref(ptr), C.byref(st)), allow=(-5,))
        return ptr.value, st.as_dict()

    def cancel(self):
        self.lib.ppg_cancel(self._h)

    def set_destination(self, destination: str):
        """scene->getDestinationFile(): with dumpSDTree=true every non-final iteration writes <destination>-NN.sdt."""
        _check(self.lib, self.lib.ppg_set_destination(self._h, destination.encode()))
        return self

    def dump_sdtree(self, path: str):
        _check(self.lib, self.lib.ppg_dump_sdtree(self._h, path.encode()))

    def op_emitter_sample_direct(self, ref, ref_n, sample, max_interactions=-1):
        """Scene::sampleAttenuatedEmitterDirect at the points `ref` of this handle's scene (ppg_op_emitter_sample_direct): (d, value, pdf, dist)."""
        f = C.POINTER(C.c_float)
        ref = np.ascontiguousarray(ref, np.float32); ref_n = np.ascontiguousarray(ref_n, np.float32); smp = np.ascontiguousarray(sample, np.float32)
        n = len(ref); d = np.zeros((n, 3), np.float32); val = np.zeros((n, 3), np.float32); pdf = np.zeros(n, np.float32); dist = np.zeros(n, np.float32)
        _check(self.lib, self.lib.ppg_op_emitter_sample_direct(self._h, n, ref.ctypes.data_as(f), ref_n.ctypes.data_as(f), smp.ctypes.data_as(f), max_interactions,
                                                               d.ctypes.data_as(f), val.ctypes.data_as(f), pdf.ctypes.data_as(f), dist.ctypes.data_as(f)))
        return d, val, pdf, dist

    def op_env_pdf(self, d):
        """(light-sampling density incl. the emitter choice, radiance) of the environment emitter for world directions `d` (ppg_op_env_pdf)."""
        f = C.POINTER(C.c_float)
        d = np.ascontiguousarray(d, np.float32); pdf = np.zeros(len(d), np.float32); val = np.zeros((len(d), 3), np.float32)
        _check(self.lib, self.lib.ppg_op_env_pdf(self._h, len(d), d.ctypes.data_as(f), pdf.ctypes.data_as(f), val.ctypes.data_as(f)))
        return pdf, val

    def moment_images(self):
        a = np.empty((self.H, self.W, 4), np.float32)
        b = np.empty_like(a)
        _check(self.lib, self.lib.ppg_get_moment_images(self._h, a.ctypes.data_as(C.POINTER(C.c_float)), b.ctypes.data_as(C.POINTER(C.c_float))))
        return a, b


def torch_allreduce(stream_sync=True):
    """Returns an allreduce callback for ``GuidedPathTracer.set_allreduce`` that runs
    ``torch.distributed.all_reduce`` (NCCL over NVLink/NVSwitch) on the library's device buffer in place."""
    import torch
    import torch.distributed as dist

    class _Ptr:
        def __init__(self, ptr, n):
            self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 3, "strides": None}

    def fn(ptr, n):
        t = torch.as_tensor(_Ptr(ptr, n), device=torch.device("cuda", torch.cuda.current_device()))
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        if stream_sync:
            torch.cuda.current_stream().synchronize()
    return fn


# ---- kernel-level operators on caller-supplied tree arrays (ppg_op_*) --------------------------------------

def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def op_dtree_pdf(sums, children, tree_first, tree_sum, tree_weight, query_tree, query_dir, device=0):
    lib = capi.load_library()
    sums = np.ascontiguousarray(sums, np.float32); children = np.ascontiguousarray(children, np.uint16)
    tf = np.ascontiguousarray(tree_first, np.uint32); ts = np.ascontiguousarray(tree_sum, np.float32); tw = np.ascontiguousarray(tree_weight, np.float32)
    qt = np.ascontiguousarray(query_tree, np.uint32); qd = np.ascontiguousarray(query_dir, np.float32)
    out = np.zeros(len(qt), np.float32)
    _check(lib, lib.ppg_op_dtree_pdf(device, _p(sums, C.c_float), _p(children, C.c_uint16), len(sums), _p(tf, C.c_uint32), _p(ts, C.c_float),
                                     _p(tw, C.c_float), len(tf), _p(qt, C.c_uint32), _p(qd, C.c_float), len(qt), _p(out, C.c_float)))
    return out


def op_dtree_sample(sums, children, tree_first, tree_sum, tree_weight, query_tree, rnd, device=0):
    lib = capi.load_library()
    sums = np.ascontiguousarray(sums, np.float32); children = np.ascontiguousarray(children, np.uint16)
    tf = np.ascontiguousarray(tree_first, np.uint32); ts = np.ascontiguousarray(tree_sum, np.float32); tw = np.ascontiguousarray(tree_weight, np.float32)
    qt = np.ascontiguousarray(query_tree, np.uint32); rnd = np.ascontiguousarray(rnd, np.float32)
    out = np.zeros((len(qt), 3), np.float32)
    _check(lib, lib.ppg_op_dtree_sample(device, _p(sums, C.c_float), _p(children, C.c_uint16), len(sums), _p(tf, C.c_uint32), _p(ts, C.c_float),
                                        _p(tw, C.c_float), len(tf), _p(qt, C.c_uint32), _p(rnd, C.c_float), rnd.shape[1], len(qt), _p(out, C.c_float)))
    return out


def op_dtree_record(sums, children, tree_first, tree_weight, rec_tree, rec_dir, rec_radiance, rec_wo_pdf, rec_weight, directional_filter=0, device=0):
    lib = capi.load_library()
    sums = np.array(sums, np.float32, copy=True, order="C"); children = np.ascontiguousarray(children, np.uint16)
    tf = np.ascontiguousarray(tree_first, np.uint32); tw = np.array(tree_weight, np.float32, copy=True, order="C")
    rt = np.ascontiguousarray(rec_tree, np.uint32); rd = np.ascontiguousarray(rec_dir, np.float32)
    rr = np.ascontiguousarray(rec_radiance, np.float32); rp = np.ascontiguousarray(rec_wo_pdf, np.float32); rw = np.ascontiguousarray(rec_weight, np.float32)
    _check(lib, lib.ppg_op_dtree_record(device, _p(sums, C.c_float), _p(children, C.c_uint16), len(sums), _p(tf, C.c_uint32), _p(tw, C.c_float), len(tf),
                                        _p(rt, C.c_uint32), _p(rd, C.c_float), _p(rr, C.c_float), _p(rp, C.c_float), _p(rw, C.c_float), len(rt), directional_filter))
    return sums, tw


def op_fraction_replay(states, rec_a, rec_b, counts, loss, cap=None, replicas=1, merge=False, device=0):
    """The renderer's sampling-fraction replay (ppg_op_fraction_replay) on given records.  states (L, 6); rec_a (n, 4) float32 with the leaf
    index's bits in column 0; rec_b (n, 2); counts (batches, replicas) records per group, stored in that order.  Returns a dict of per-batch
    arrays: states (B, L, 6), replicas (B, R, L, 6), theta (B, L), sorted_a / sorted_b (the bucketed lists, rec_a / rec_b layout), progress (B, 2)."""
    lib = capi.load_library()
    st = np.ascontiguousarray(states, np.float32); ra = np.ascontiguousarray(rec_a, np.float32).reshape(-1, 4); rb = np.ascontiguousarray(rec_b, np.float32).reshape(-1, 2)
    cnt = np.ascontiguousarray(np.asarray(counts, np.uint64).reshape(-1, replicas), np.uint64)
    B, L = cnt.shape[0], len(st)
    assert int(cnt.sum()) == len(ra) == len(rb)
    cap = int(cap if cap is not None else max(int(cnt.max()), 1))
    out = dict(states=np.zeros((B, L, 6), np.float32), replicas=np.zeros((B, replicas, L, 6), np.float32), theta=np.zeros((B, L), np.float32),
               sorted_a=np.zeros_like(ra), sorted_b=np.zeros_like(rb), progress=np.zeros((B, 2), np.uint64))
    code = {"kl": 1, "var": 2}[loss] if isinstance(loss, str) else int(loss)
    _check(lib, lib.ppg_op_fraction_replay(device, _p(st, C.c_float), L, _p(ra, C.c_float), _p(rb, C.c_float), _p(cnt, C.c_size_t), B, replicas, int(merge), cap, code,
                                           _p(out["states"], C.c_float), _p(out["replicas"], C.c_float), _p(out["theta"], C.c_float),
                                           _p(out["sorted_a"], C.c_float), _p(out["sorted_b"], C.c_float), _p(out["progress"], C.c_ulonglong)))
    return out


def op_bvh_build(positions, indices, threads=0):
    """The BVH ppg_set_scene builds, on the host (no device): (nodes (N,8) float32, order (T,) uint32, max depth, milliseconds)."""
    lib = capi.load_library()
    pos = np.ascontiguousarray(positions, np.float32); idx = np.ascontiguousarray(indices, np.uint32)
    nt = len(idx); nodes = np.zeros((2 * nt + 1, 8), np.float32); order = np.zeros(nt, np.uint32)
    n = C.c_size_t(); depth = C.c_int(); ms = C.c_double()
    _check(lib, lib.ppg_op_bvh_build(_p(pos, C.c_float), _p(idx, C.c_uint32), nt, threads, _p(nodes, C.c_float), len(nodes), _p(order, C.c_uint32),
                                     C.byref(n), C.byref(depth), C.byref(ms)))
    return nodes[:n.value], order, depth.value, ms.value


def op_stree_lookup(node_children, aabb_min, aabb_extent, points, device=0):
    lib = capi.load_library()
    nc = np.ascontiguousarray(node_children, np.uint32); pts = np.ascontiguousarray(points, np.float32)
    mn = np.ascontiguousarray(aabb_min, np.float32); ex = np.ascontiguousarray(aabb_extent, np.float32)
    leaf = np.zeros(len(pts), np.uint32); size = np.zeros((len(pts), 3), np.float32)
    _check(lib, lib.ppg_op_stree_lookup(device, _p(nc, C.c_uint32), len(nc), _p(mn, C.c_float), _p(ex, C.c_float), _p(pts, C.c_float), len(pts),
                                        _p(leaf, C.c_uint32), _p(size, C.c_float)))
    return leaf, size
