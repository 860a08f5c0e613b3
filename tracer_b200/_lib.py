"""ctypes binding of libtracer_rq.so (include/tracer_rq.h, include/tracer_rq_harness.h).

The library is built in-tree by `__graft_entry__.build()` / `make -C tracer_b200/csrc`. There is no
Python or CPU fallback: if the shared object is missing, importing this module raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# TRQ_LIB: developer override (instrumented builds from tools/build_variant.sh); the product library otherwise
LIB_PATH = os.environ.get("TRQ_LIB") or os.path.join(_HERE, "libtracer_rq.so")

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "or `make -C tracer_b200/csrc`. tracer_b200 has no CPU / pure-Python fallback."
    )

lib = C.CDLL(LIB_PATH)

OK, ERR_INVALID, ERR_LAYOUT, ERR_DEPTH, ERR_CUDA, ERR_NOMEM, ERR_NO_DEVICE = 0, -1, -2, -3, -4, -5, -6


class SceneDesc(C.Structure):
    _fields_ = [
        ("sphereList", C.c_void_p), ("nSphere", C.c_uint32),
        ("squareList", C.c_void_p), ("nSquare", C.c_uint32),
        ("cubeList", C.c_void_p), ("nCube", C.c_uint32),
        ("triList", C.c_void_p), ("nVert", C.c_uint32),
        ("idxList", C.c_void_p), ("nTri", C.c_uint32),
        ("bvhList", C.c_void_p), ("nNode", C.c_uint32),
    ]


class SceneInfo(C.Structure):
    _fields_ = [
        ("nNode", C.c_uint32), ("nInterior", C.c_uint32), ("nLeaf", C.c_uint32), ("maxDepth", C.c_uint32),
        ("nTri", C.c_uint32), ("nSphere", C.c_uint32), ("nSquare", C.c_uint32), ("nCube", C.c_uint32),
        ("bytesReferenceLayout", C.c_uint64), ("bytesPacked", C.c_uint64),
        ("device", C.c_int32), ("topNodes", C.c_uint32),
    ]


class Camera(C.Structure):
    _fields_ = [("lookFrom", C.c_float * 3), ("lookAt", C.c_float * 3), ("viewUp", C.c_float * 3),
                ("vfov", C.c_float), ("aspect", C.c_float), ("aperture", C.c_float), ("focus_dist", C.c_float)]


# every symbol include/*.h declares; tests/test_abi.py checks the library exports all of them
ABI_SYMBOLS = [
    "trq_version", "trq_last_error_string", "trq_device_count",
    "trq_scene_create", "trq_scene_create_device", "trq_scene_update_vertices", "trq_scene_update_primitives", "trq_scene_rebuild", "trq_scene_copy_bvh", "trq_scene_destroy", "trq_device_trim", "trq_scene_info",
    "trq_kernel_config_count", "trq_kernel_config_name", "trq_scene_set_kernel_config", "trq_scene_kernel_config",
    "trq_trace", "trq_host_sync", "trq_expand_hits", "trq_launch_count", "trq_profile_enable", "trq_profile_read", "trq_probe_bandwidth",
    "trq_bvh_build_node", "trq_bvh_build_nodes_triangles", "trq_bvh_build_nodes_triangles_device", "trq_bvh_build_nodes_device", "trq_bvh_build_tree", "trq_bvh_build_tree_gpu", "trq_bvh_build_tree_device",
    "trq_bvh_build_tree_morton", "trq_bvh_build_tree_morton_device",
    "trq_cast_rays", "trq_trace_indirect", "trq_spawn_bounce", "trq_spawn_shadow", "trq_spawn_bounce_rng", "trq_spawn_shadow_rng", "trq_rng_frame_begin",
    "trq_mgpu_create", "trq_mgpu_device_count", "trq_mgpu_scene", "trq_mgpu_shard", "trq_mgpu_trace", "trq_mgpu_destroy",
    "trq_gather_create", "trq_gather_connect", "trq_trace_gather", "trq_gather_wait", "trq_gather_status", "trq_gather_destroy",
]
HARNESS_SYMBOLS = [
    "trqh_pcg32_fill_f32", "trqh_pcg32_fill_u32", "trqh_normalize_rays", "trqh_offset_ray",
    "trqh_make_soup", "trqh_gen_random_rays", "trqh_make_camera", "trqh_gen_camera_rays",
    "trqh_gen_bounce_rays", "trqh_gen_shadow_rays", "trqh_gen_bounce_rays_rng", "trqh_gen_shadow_rays_rng", "trqh_rng_frame_begin",
]

_vp, _u32, _u64, _i32, _f32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int32, C.c_float

lib.trq_version.restype = C.c_int
lib.trq_last_error_string.restype = C.c_char_p
lib.trq_device_count.restype = C.c_int
lib.trq_launch_count.restype = _u64
lib.trq_scene_create.argtypes = [C.POINTER(SceneDesc), C.c_int, C.POINTER(_vp)]
lib.trq_scene_create_device.argtypes = [C.POINTER(SceneDesc), C.c_int, C.POINTER(_vp)]
lib.trq_scene_update_vertices.argtypes = [_vp, _vp, _u32, _u32]
lib.trq_scene_update_primitives.argtypes = [_vp, C.POINTER(SceneDesc), _u32]
lib.trq_scene_rebuild.argtypes = [_vp, _vp, _u32, _u32]
lib.trq_scene_copy_bvh.argtypes = [_vp, _vp, _u32]
lib.trq_scene_destroy.argtypes = [_vp]
lib.trq_device_trim.argtypes = [C.c_int]
lib.trq_scene_info.argtypes = [_vp, C.POINTER(SceneInfo)]
lib.trq_kernel_config_name.argtypes = [C.c_int]
lib.trq_kernel_config_name.restype = C.c_char_p
lib.trq_scene_set_kernel_config.argtypes = [_vp, C.c_int, C.POINTER(_u32)]
lib.trq_scene_kernel_config.argtypes = [_vp]
lib.trq_trace.argtypes = [_vp, _vp, _u64, _u32, _vp, _vp]
lib.trq_host_sync.argtypes = [_vp]
lib.trq_expand_hits.argtypes = [_vp, _vp, _vp, _u64, _u32, _vp, _vp]
lib.trq_probe_bandwidth.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_double)]
lib.trq_profile_enable.argtypes = [_vp, C.c_int]
lib.trq_profile_read.argtypes = [_vp, C.POINTER(_u32), C.POINTER(_f32), C.POINTER(_f32)]
lib.trq_mgpu_create.argtypes = [C.POINTER(SceneDesc), _vp, C.c_int, C.POINTER(_vp)]
lib.trq_mgpu_device_count.argtypes = [_vp]
lib.trq_mgpu_scene.argtypes = [_vp, C.c_int]
lib.trq_mgpu_scene.restype = _vp
lib.trq_mgpu_shard.argtypes = [_vp, _u64, C.c_int, C.POINTER(_u64), C.POINTER(_u64)]
lib.trq_mgpu_trace.argtypes = [_vp, _vp, _u64, _u32, _vp]
lib.trq_mgpu_destroy.argtypes = [_vp]
lib.trq_gather_create.argtypes = [_vp, _u32, _u32, _u64, C.POINTER(_vp), _vp]
lib.trq_gather_connect.argtypes = [_vp, _vp]
lib.trq_trace_gather.argtypes = [_vp, _vp, _vp, _u64, _u32, _vp]
lib.trq_gather_wait.argtypes = [_vp, _vp, C.POINTER(_vp), C.POINTER(_vp)]
lib.trq_gather_status.argtypes = [_vp]
lib.trq_gather_destroy.argtypes = [_vp]
lib.trq_cast_rays.argtypes = [_vp, C.POINTER(Camera), _u32, _u32, _vp, _vp]
lib.trq_trace_indirect.argtypes = [_vp, _vp, _vp, _u64, _u32, _vp, _vp]
lib.trq_spawn_bounce.argtypes = [_vp, _vp, _vp, _u64, _vp, _u64, _vp, _vp, _vp, _vp]
lib.trq_spawn_shadow.argtypes = [_vp, _vp, _vp, _u64, _vp, _u64, _u32, _u32, _vp, _vp, _vp, _vp]
lib.trq_rng_frame_begin.argtypes = [_vp, _vp, _u64, _vp]
lib.trqh_rng_frame_begin.argtypes = [_vp, _u64]
lib.trqh_rng_frame_begin.restype = None
lib.trq_spawn_bounce_rng.argtypes = [_vp, _vp, _vp, _u64, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp]
lib.trq_spawn_shadow_rng.argtypes = [_vp, _vp, _vp, _u64, _vp, _u64, _vp, _vp, _u32, _u32, _vp, _vp, _vp, _vp]
lib.trq_bvh_build_node.argtypes = [_vp, _vp, _vp, _i32, _u32, _vp]
lib.trq_bvh_build_nodes_triangles.argtypes = [_vp, _vp, _u32, _u32, _vp]
lib.trq_bvh_build_nodes_triangles_device.argtypes = [_vp, _vp, _u32, _u32, _vp, C.c_int, _vp]
lib.trq_bvh_build_nodes_device.argtypes = [_i32, _vp, _u32, _u32, _vp, C.c_int, _vp]
lib.trq_bvh_build_tree.argtypes = [_vp, _u32, C.POINTER(_u32), C.POINTER(_u32)]
lib.trq_bvh_build_tree_gpu.argtypes = [_vp, _u32, C.c_int, C.POINTER(_u32), C.POINTER(_u32)]
lib.trq_bvh_build_tree_device.argtypes = [_vp, _u32, C.c_int, C.POINTER(_u32), C.POINTER(_u32)]
lib.trq_bvh_build_tree_morton.argtypes = [_vp, _u32, C.POINTER(_u32), C.POINTER(_u32)]
lib.trq_bvh_build_tree_morton_device.argtypes = [_vp, _u32, C.c_int, C.POINTER(_u32), C.POINTER(_u32)]

lib.trqh_pcg32_fill_f32.argtypes = [_u64, _u64, _u64, _vp]
lib.trqh_pcg32_fill_f32.restype = None
lib.trqh_pcg32_fill_u32.argtypes = [_u64, _u64, _u64, _vp]
lib.trqh_pcg32_fill_u32.restype = None
lib.trqh_normalize_rays.argtypes = [_vp, _u64]
lib.trqh_normalize_rays.restype = None
lib.trqh_offset_ray.argtypes = [_vp, _vp, _vp]
lib.trqh_offset_ray.restype = None
lib.trqh_make_soup.argtypes = [_u32, _u64, _f32, _vp, _vp]
lib.trqh_make_soup.restype = None
lib.trqh_gen_random_rays.argtypes = [_u64, _u64, _u64, _vp, _vp, _f32, _vp]
lib.trqh_gen_random_rays.restype = None
lib.trqh_make_camera.argtypes = [_vp, _vp, _vp, _f32, _f32, _f32, _vp]
lib.trqh_make_camera.restype = None
lib.trqh_gen_camera_rays.argtypes = [_vp, _vp, _vp, _f32, _f32, _f32, _u32, _u32, _vp]
lib.trqh_gen_camera_rays.restype = None
lib.trqh_gen_bounce_rays.argtypes = [_vp, _u64, _u64, _vp, _vp]
lib.trqh_gen_bounce_rays.restype = _u64
lib.trqh_gen_shadow_rays.argtypes = [_vp, _u64, _u64, _vp, _vp, _vp, _vp]
lib.trqh_gen_shadow_rays.restype = _u64
lib.trqh_gen_bounce_rays_rng.argtypes = [_vp, _u64, _u64, _vp, _vp, _vp, _vp]
lib.trqh_gen_bounce_rays_rng.restype = _u64
lib.trqh_gen_shadow_rays_rng.argtypes = [_vp, _u64, _u64, _vp, _vp, _vp, _vp, _vp, _vp]
lib.trqh_gen_shadow_rays_rng.restype = _u64


class TrqError(RuntimeError):
    def __init__(self, status, where):
        self.status = status
        msg = lib.trq_last_error_string()
        super().__init__(f"{where}: status {status}: {msg.decode() if msg else ''}")


def check(status, where):
    if status != OK:
        raise TrqError(status, where)
