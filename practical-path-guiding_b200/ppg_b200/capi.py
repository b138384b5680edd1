"""ctypes mirror of include/ppg.h (the C ABI of libppg_b200.so).

This is the reference-side binding a Python host would add; the structs are
laid out exactly as in the header.  The library is loaded lazily and loudly:
there is no fallback if the CUDA extension is missing.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

PPG_MAX_ITERATIONS = 40
PPG_KERNEL_CLASSES = 8
KERNEL_CLASSES = ["bounce", "commit", "film", "refine", "reset", "build", "adam", "other"]

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PPG_B200_LIB") or os.path.join(os.path.dirname(_HERE), "csrc", "libppg_b200.so")   # PPG_B200_LIB: A/B builds of the same CUDA sources


class PpgParams(C.Structure):
    _fields_ = [
        ("nee", C.c_int32), ("sample_combination", C.c_int32), ("spatial_filter", C.c_int32),
        ("directional_filter", C.c_int32), ("bsdf_sampling_fraction_loss", C.c_int32),
        ("sd_tree_max_memory", C.c_int32), ("s_tree_threshold", C.c_int32), ("d_tree_threshold", C.c_float),
        ("bsdf_sampling_fraction", C.c_float), ("spp_per_pass", C.c_int32), ("budget_type", C.c_int32),
        ("budget", C.c_float), ("dump_sd_tree", C.c_int32), ("max_depth", C.c_int32), ("rr_depth", C.c_int32),
        ("strict_normals", C.c_int32), ("hide_emitters", C.c_int32), ("seed", C.c_uint64),
    ]


class PpgBsdf(C.Structure):
    _fields_ = [("type", C.c_int32), ("flags", C.c_uint32), ("reflectance", C.c_float * 3), ("specular_transmittance", C.c_float * 3),
                ("eta", C.c_float * 3), ("k", C.c_float * 3), ("alpha", C.c_float), ("distribution", C.c_int32),
                ("specular_reflectance", C.c_float * 3), ("fdr_int", C.c_float), ("specular_sampling_weight", C.c_float), ("table", C.c_int32), ("opacity", C.c_float * 3),
                ("reflectance_texture", C.c_uint32), ("bump_texture", C.c_uint32), ("reserved", C.c_uint32)]


class PpgTexture(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("channels", C.c_uint32), ("wrap_u", C.c_uint32), ("wrap_v", C.c_uint32),
                ("uv_scale", C.c_float * 2), ("uv_offset", C.c_float * 2), ("reserved", C.c_uint32), ("first_texel", C.c_uint64)]


class PpgEnvmap(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("texels", C.POINTER(C.c_uint16)), ("scale", C.c_float), ("world_to_env", C.c_float * 9)]


class PpgShape(C.Structure):
    _fields_ = [("first_triangle", C.c_uint32), ("n_triangles", C.c_uint32), ("bsdf", C.c_int32), ("emitter", C.c_int32),
                ("has_normals", C.c_uint32), ("has_uvs", C.c_uint32), ("reserved", C.c_uint32 * 2)]


class PpgSphere(C.Structure):
    _fields_ = [("center", C.c_float * 3), ("radius", C.c_float), ("shape", C.c_int32), ("flip_normals", C.c_int32)]


class PpgCamera(C.Structure):
    _fields_ = [("to_world", C.c_float * 16), ("x_fov_deg", C.c_float), ("near_clip", C.c_float), ("far_clip", C.c_float),
                ("film_width", C.c_int32), ("film_height", C.c_int32)]


class PpgSceneDesc(C.Structure):
    _fields_ = [
        ("n_vertices", C.c_uint32), ("n_triangles", C.c_uint32), ("n_shapes", C.c_uint32), ("n_bsdfs", C.c_uint32),
        ("n_emitters", C.c_uint32),
        ("positions", C.POINTER(C.c_float)), ("normals", C.POINTER(C.c_float)), ("uvs", C.POINTER(C.c_float)),
        ("indices", C.POINTER(C.c_uint32)), ("triangle_shape", C.POINTER(C.c_uint32)),
        ("shapes", C.POINTER(PpgShape)), ("bsdfs", C.POINTER(PpgBsdf)), ("area_radiance", C.POINTER(C.c_float)),
        ("bsdf_tables", C.POINTER(C.c_float)), ("n_bsdf_tables", C.c_uint32),
        ("n_spheres", C.c_uint32), ("spheres", C.POINTER(PpgSphere)),
        ("camera", PpgCamera), ("aabb_min", C.c_float * 3), ("aabb_max", C.c_float * 3),
        ("n_textures", C.c_uint32), ("reserved", C.c_uint32), ("textures", C.POINTER(PpgTexture)), ("texels", C.POINTER(C.c_uint16)),
        ("n_texels", C.c_uint64), ("envmap", PpgEnvmap),
    ]


class PpgIterationStats(C.Structure):
    _fields_ = [
        ("iteration", C.c_int32), ("passes", C.c_int32), ("is_final", C.c_int32), ("total_passes", C.c_int32),
        ("seconds", C.c_float), ("variance", C.c_float), ("reset_seconds", C.c_float), ("build_seconds", C.c_float),
        ("depth_min", C.c_int32), ("depth_max", C.c_int32), ("depth_avg", C.c_float),
        ("mean_radiance_min", C.c_float), ("mean_radiance_avg", C.c_float), ("mean_radiance_max", C.c_float),
        ("nodes_min", C.c_uint64), ("nodes_max", C.c_uint64), ("nodes_avg", C.c_float),
        ("weight_min", C.c_float), ("weight_avg", C.c_float), ("weight_max", C.c_float),
        ("s_tree_nodes", C.c_uint32), ("s_tree_leaves", C.c_uint32), ("s_tree_depth_avg", C.c_double),
        ("vertices", C.c_uint64), ("paths", C.c_uint64), ("recorded_vertices", C.c_uint64),
    ]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class PpgStats(C.Structure):
    _fields_ = [
        ("n_iterations", C.c_int32), ("total_passes", C.c_int32), ("total_paths", C.c_uint64), ("total_vertices", C.c_uint64),
        ("render_seconds", C.c_double), ("device_seconds", C.c_double), ("final_variance", C.c_double),
        ("kernel_launches", C.c_uint64), ("kernel_ms", C.c_double * PPG_KERNEL_CLASSES), ("kernel_count", C.c_uint64 * PPG_KERNEL_CLASSES),
        ("render_device_ms", C.c_double), ("truncated_paths", C.c_uint64), ("dropped_records", C.c_uint64), ("sub_batches", C.c_uint64), ("invalid_rays", C.c_uint64), ("iterations", PpgIterationStats * PPG_MAX_ITERATIONS),
    ]

    def as_dict(self):
        d = {n: getattr(self, n) for n, _ in self._fields_ if n not in ("iterations", "kernel_ms", "kernel_count")}
        d["kernel_ms"] = {k: self.kernel_ms[i] for i, k in enumerate(KERNEL_CLASSES)}
        d["kernel_count"] = {k: self.kernel_count[i] for i, k in enumerate(KERNEL_CLASSES)}
        d["iterations"] = [self.iterations[i].as_dict() for i in range(self.n_iterations)]
        return d


ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t)
CLOCK_FN = C.CFUNCTYPE(C.c_double, C.c_void_p)
FILM_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int)


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _up(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint32))


class SceneArrays:
    """Owns contiguous numpy arrays + the ppg_scene_desc pointing into them."""

    def __init__(self, scene):
        self.positions = np.ascontiguousarray(scene.positions, np.float32)
        self.normals = np.ascontiguousarray(scene.normals, np.float32)
        self.uvs = np.ascontiguousarray(scene.uvs, np.float32)
        self.indices = np.ascontiguousarray(scene.indices, np.uint32)
        self.triangle_shape = np.ascontiguousarray(scene.triangle_shape, np.uint32)
        self.shapes = np.ascontiguousarray(scene.shapes, np.int32)          # (S,8) == ppg_shape
        b = np.asarray(scene.bsdfs, np.float32)
        if b.shape[1] < 28:                                                   # arrays written before the struct grew to 112 bytes
            b = np.concatenate([b, np.zeros((len(b), 28 - b.shape[1]), np.float32)], axis=1)
        self.bsdfs = np.ascontiguousarray(b, np.float32)                    # (B,28) == ppg_bsdf
        tables = getattr(scene, "bsdf_tables", None)
        self.tables = np.ascontiguousarray(tables if tables is not None and len(tables) else np.zeros((0, 100)), np.float32)
        self.radiance = np.ascontiguousarray(scene.area_radiance, np.float32)
        sph = getattr(scene, "spheres", None)
        self.spheres = np.ascontiguousarray(sph if sph is not None and len(sph) else np.zeros((0, 6)), np.float32)   # (K,6) == ppg_sphere
        d = PpgSceneDesc()
        d.n_vertices = len(self.positions); d.n_triangles = len(self.indices); d.n_shapes = len(self.shapes)
        d.n_bsdfs = len(self.bsdfs); d.n_emitters = len(self.radiance)
        d.positions = _fp(self.positions); d.normals = _fp(self.normals); d.uvs = _fp(self.uvs)
        d.indices = _up(self.indices); d.triangle_shape = _up(self.triangle_shape)
        d.shapes = self.shapes.ctypes.data_as(C.POINTER(PpgShape))
        d.bsdfs = self.bsdfs.ctypes.data_as(C.POINTER(PpgBsdf))
        d.area_radiance = _fp(self.radiance)
        d.bsdf_tables = _fp(self.tables) if len(self.tables) else None
        d.n_bsdf_tables = len(self.tables)
        d.n_spheres = len(self.spheres)
        d.spheres = self.spheres.ctypes.data_as(C.POINTER(PpgSphere)) if len(self.spheres) else None
        cam = PpgCamera()
        m = np.ascontiguousarray(scene.cam_to_world, np.float32).reshape(16)
        for i in range(16):
            cam.to_world[i] = float(m[i])
        cam.x_fov_deg = scene.x_fov_deg; cam.near_clip = scene.near_clip; cam.far_clip = scene.far_clip
        cam.film_width = scene.film_width; cam.film_height = scene.film_height
        d.camera = cam
        for i in range(3):
            d.aabb_min[i] = float(scene.aabb_min[i]); d.aabb_max[i] = float(scene.aabb_max[i])
        tex = getattr(scene, "textures", None)
        if tex is not None and len(tex):
            self.textures = np.ascontiguousarray(tex)                           # TEXTURE_DTYPE == ppg_texture
            self.texels = np.ascontiguousarray(scene.texels, np.uint16)
            assert self.textures.dtype.itemsize == C.sizeof(PpgTexture)
            d.n_textures = len(self.textures); d.textures = self.textures.ctypes.data_as(C.POINTER(PpgTexture))
            d.texels = self.texels.ctypes.data_as(C.POINTER(C.c_uint16)); d.n_texels = len(self.texels)
        env = getattr(scene, "envmap", None)
        if env:
            self.env_texels = np.ascontiguousarray(env["texels"], np.uint16)
            d.envmap.height, d.envmap.width = self.env_texels.shape[:2]
            d.envmap.texels = self.env_texels.ctypes.data_as(C.POINTER(C.c_uint16)); d.envmap.scale = float(env["scale"])
            m = np.asarray(env["world_to_env"], np.float32).reshape(9)
            for i in range(9):
                d.envmap.world_to_env[i] = float(m[i])
        self.desc = d


_lib = None


def load_library(path: str | None = None):
    """dlopen libppg_b200.so and declare the prototypes of include/ppg.h.  Raises if the CUDA extension is not built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise RuntimeError(f"{p} not found: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()'). "
                           "There is no CPU fallback.")
    lib = C.CDLL(p)
    H = C.c_void_p
    lib.ppg_description.restype = C.c_char_p
    lib.ppg_last_error.restype = C.c_char_p
    lib.ppg_abi_version.restype = C.c_int
    lib.ppg_params_default.argtypes = [C.POINTER(PpgParams)]; lib.ppg_params_default.restype = None
    lib.ppg_params_set.argtypes = [C.POINTER(PpgParams), C.c_char_p, C.c_char_p]
    lib.ppg_params_validate.argtypes = [C.POINTER(PpgParams)]
    lib.ppg_create.argtypes = [C.POINTER(PpgParams), C.c_int, C.POINTER(H)]
    lib.ppg_destroy.argtypes = [H]; lib.ppg_destroy.restype = None
    lib.ppg_set_scene.argtypes = [H, C.POINTER(PpgSceneDesc)]
    lib.ppg_scene_file_load.argtypes = [C.c_char_p, C.POINTER(PpgSceneDesc), C.POINTER(C.c_void_p), C.POINTER(C.c_char_p)]
    lib.ppg_scene_file_free.argtypes = [C.c_void_p]; lib.ppg_scene_file_free.restype = None
    lib.ppg_set_shard.argtypes = [H, C.c_int, C.c_int]
    lib.ppg_set_allreduce.argtypes = [H, ALLREDUCE_FN, C.c_void_p]
    lib.ppg_nccl_unique_id.argtypes = [C.c_void_p]
    lib.ppg_nccl_init.argtypes = [H, C.c_void_p, C.c_int, C.c_int]
    lib.ppg_set_clock.argtypes = [H, CLOCK_FN, C.c_void_p]
    lib.ppg_set_film_callback.argtypes = [H, FILM_FN, C.c_void_p]
    lib.ppg_render.argtypes = [H, C.POINTER(C.c_float), C.POINTER(PpgStats)]
    lib.ppg_render_device.argtypes = [H, C.POINTER(C.c_void_p), C.POINTER(PpgStats)]
    lib.ppg_cancel.argtypes = [H]
    lib.ppg_copy_from_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    lib.ppg_dump_sdtree.argtypes = [H, C.c_char_p]
    lib.ppg_set_destination.argtypes = [H, C.c_char_p]
    lib.ppg_get_moment_images.argtypes = [H, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    u16p = C.POINTER(C.c_uint16); u32p = C.POINTER(C.c_uint32); f32p = C.POINTER(C.c_float)
    lib.ppg_op_dtree_pdf.argtypes = [C.c_int, f32p, u16p, C.c_size_t, u32p, f32p, f32p, C.c_size_t, u32p, f32p, C.c_size_t, f32p]
    lib.ppg_op_dtree_sample.argtypes = [C.c_int, f32p, u16p, C.c_size_t, u32p, f32p, f32p, C.c_size_t, u32p, f32p, C.c_size_t, C.c_size_t, f32p]
    lib.ppg_op_dtree_record.argtypes = [C.c_int, f32p, u16p, C.c_size_t, u32p, f32p, C.c_size_t, u32p, f32p, f32p, f32p, f32p, C.c_size_t, C.c_int]
    lib.ppg_op_fraction_replay.argtypes = [C.c_int, f32p, C.c_size_t, f32p, f32p, C.POINTER(C.c_size_t), C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_int,
                                           f32p, f32p, f32p, f32p, f32p, C.POINTER(C.c_ulonglong)]
    lib.ppg_op_stree_lookup.argtypes = [C.c_int, u32p, C.c_size_t, f32p, f32p, f32p, C.c_size_t, u32p, f32p]
    lib.ppg_op_bvh_build.argtypes = [f32p, u32p, C.c_size_t, C.c_int, f32p, C.c_size_t, u32p, C.POINTER(C.c_size_t), C.POINTER(C.c_int), C.POINTER(C.c_double)]
    lib.ppg_op_emitter_sample_direct.argtypes = [H, C.c_size_t, f32p, f32p, f32p, C.c_int, f32p, f32p, f32p, f32p]
    lib.ppg_op_env_pdf.argtypes = [H, C.c_size_t, f32p, f32p, f32p]
    if path is None:
        _lib = lib
    return lib


EXPORTED_SYMBOLS = [
    "ppg_params_default", "ppg_params_set", "ppg_params_validate", "ppg_description", "ppg_abi_version", "ppg_create",
    "ppg_destroy", "ppg_scene_file_load", "ppg_scene_file_free", "ppg_set_scene", "ppg_set_shard", "ppg_set_allreduce", "ppg_nccl_unique_id", "ppg_nccl_init", "ppg_set_clock", "ppg_set_film_callback", "ppg_render", "ppg_render_device", "ppg_cancel",
    "ppg_copy_from_device", "ppg_dump_sdtree", "ppg_set_destination", "ppg_get_moment_images", "ppg_last_error", "ppg_op_dtree_pdf", "ppg_op_dtree_sample",
    "ppg_op_dtree_record", "ppg_op_fraction_replay", "ppg_op_stree_lookup", "ppg_op_emitter_sample_direct", "ppg_op_env_pdf", "ppg_op_bvh_build",
]
