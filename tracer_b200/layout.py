"""numpy dtypes for the reference byte layouts and the C-ABI ray / hit structs.

Sizes are the reference's own (Metal / Apple-simd rules, float3 = 16 B), checked against the
verbatim build of the reference headers in tests/test_layout.py:
  BVH 64 B            RT_Metal/Metal/BVH.hh:15-22
  TriangleVertex 32 B RT_Metal/Metal/Triangle.hh:12-18
  Sphere 272 B        RT_Metal/Metal/Sphere.hh:6-15
  Square 272 B        RT_Metal/Metal/Square.hh:12-27
  Cube 240 B          RT_Metal/Metal/Cube.hh:6-13
  trq_ray / trq_hit / trq_hit_record   include/tracer_rq.h
"""
import numpy as np

# enum struct PrimitiveType  (BVH.hh:6-8)
SPHERE, SQUARE, CUBE, TRIANGLE, BVH, UNKNOW = 0, 1, 2, 3, 4, 5

AABB_FIELDS = [("mini", "<f4", 3), ("pad0", "<f4"), ("maxi", "<f4", 3), ("pad1", "<f4")]

bvh_dtype = np.dtype([
    ("parent", "<u4"), ("left", "<u4"), ("right", "<u4"), ("axis", "<u4"),
    ("pType", "<i4"), ("pIndex", "<u4"), ("pad", "<u4", 2),
    ("mini", "<f4", 3), ("pad0", "<f4"), ("maxi", "<f4", 3), ("pad1", "<f4"),
])

vertex_dtype = np.dtype([("v", "<f4", 3), ("n", "<f4", 3), ("uv", "<f4", 2)])

sphere_dtype = np.dtype([
    ("radius", "<f4"), ("pad0", "<f4", 3),
    ("center", "<f4", 3), ("pad1", "<f4"),
    ("model", "<f4", 16), ("normal", "<f4", 16), ("inverse", "<f4", 16),
    ("material", "<u4"), ("pad2", "<u4", 3),
    ("box_mini", "<f4", 3), ("pad3", "<f4"), ("box_maxi", "<f4", 3), ("pad4", "<f4"),
])

square_dtype = np.dtype([
    ("axis_i", "u1"), ("axis_j", "u1"), ("pad0", "u1", 6),
    ("range_i", "<f4", 2), ("range_j", "<f4", 2),
    ("axis_k", "u1"), ("pad1", "u1", 3), ("value_k", "<f4"),
    ("model", "<f4", 16), ("normal", "<f4", 16), ("inverse", "<f4", 16),
    ("material", "<u4"), ("pad2", "<u4", 3),
    ("box_mini", "<f4", 3), ("pad3", "<f4"), ("box_maxi", "<f4", 3), ("pad4", "<f4"),
])

cube_dtype = np.dtype([
    ("model", "<f4", 16), ("normal", "<f4", 16), ("inverse", "<f4", 16),
    ("box_mini", "<f4", 3), ("pad0", "<f4"), ("box_maxi", "<f4", 3), ("pad1", "<f4"),
    ("material", "<u4"), ("pad2", "<u4", 3),
])

ray_dtype = np.dtype([("o", "<f4", 3), ("tmax", "<f4"), ("d", "<f4", 3), ("flags", "<u4")])

hit_dtype = np.dtype([
    ("t", "<f4"), ("pType", "<u4"), ("pIndex", "<u4"), ("leafNode", "<u4"),
    ("u", "<f4"), ("v", "<f4"), ("material", "<u4"), ("flags", "<u4"),
])

# trq_hit16: id = 0xffffffff on a miss, else front << 31 | pType << 28 | pIndex
hit16_dtype = np.dtype([("t", "<f4"), ("id", "<u4"), ("u", "<f4"), ("v", "<f4")])
HIT16_MISS = 0xFFFFFFFF

record_dtype = np.dtype([
    ("hit", "<u4"), ("t", "<f4"), ("p", "<f4", 3), ("gn", "<f4", 3), ("sn", "<f4", 3),
    ("uv", "<f4", 2), ("front", "<u4"), ("material", "<u4"), ("pad", "<u4"),
])

assert bvh_dtype.itemsize == 64 and vertex_dtype.itemsize == 32
assert sphere_dtype.itemsize == 272 and square_dtype.itemsize == 272 and cube_dtype.itemsize == 240
assert ray_dtype.itemsize == 32 and hit_dtype.itemsize == 32 and hit16_dtype.itemsize == 16 and record_dtype.itemsize == 64

HIT_FLAG_HIT, HIT_FLAG_FRONT = 1, 2
TRACE_ANY, HOST_PTRS, KERNEL_REFLAYOUT, SORT_RAYS, HOST_ASYNC, HIT16, NO_SORT = 0x1, 0x2, 0x4, 0x8, 0x10, 0x20, 0x40
BUILD_MORTON = 0x80                    # trq_scene_rebuild: the Morton builder builds the new topology

FLT_MAX = float(np.finfo(np.float32).max)
FLT_MIN = float(np.finfo(np.float32).tiny)

IDENTITY4 = np.eye(4, dtype=np.float32).reshape(16)   # column-major == row-major for identity


def pack_hit16(hits):
    """hit_dtype array -> the hit16_dtype array TRQ_HIT16 produces for the same rays (host restatement, for tests)."""
    out = np.zeros(hits.shape, dtype=hit16_dtype)
    hit = (hits["flags"] & HIT_FLAG_HIT) != 0
    front = ((hits["flags"] & HIT_FLAG_FRONT) != 0).astype(np.uint32)
    out["t"], out["u"], out["v"] = hits["t"], hits["u"], hits["v"]
    out["id"] = np.where(hit, (front << 31) | (hits["pType"].astype(np.uint32) << 28) | (hits["pIndex"] & 0x0FFFFFFF), HIT16_MISS)
    return out
