"""Shared helpers for the test suite."""
import os

import numpy as np

from tracer_b200 import layout as L
from tracer_b200.scene import Primitive

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rq_golden.npz")
FIELDS = ("sphereList", "squareList", "cubeList", "triList", "idxList", "bvhList")
CASES = ("cornell_primary", "cornell_bounce", "cornell_shadow_any", "soup_closest", "soup_any_tmax",
         "icosphere_ties", "c1_spheres", "one_leaf", "two_leaves")

_cache = {}


def golden():
    if "z" not in _cache:
        _cache["z"] = np.load(GOLDEN)
    return _cache["z"]


def golden_case(name):
    """-> (Primitive, rays, any, reference records)"""
    z = golden()
    prim = Primitive(**{k: z[f"{name}/{k}"] for k in FIELDS})
    return prim, z[f"{name}/rays"], bool(z[f"{name}/any"][0]), z[f"{name}/records"]


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def refit_on_host(prim, verts):
    """trq_scene_update_vertices restated with numpy, for a tree in any node numbering: triangle leaf boxes from the
    moved vertices (trq_bvh_build_nodes_triangles), then the interior nodes reachable from the root, deepest first, as
    unions of their children. Nodes the root does not reach keep their boxes. -> the refit Primitive."""
    from tracer_b200._lib import check, lib
    nodes = prim.bvhList.copy()
    depth = np.full(nodes.size, -1, dtype=np.int64)
    depth[0] = 0
    stack = [0]
    while stack:
        i = stack.pop()
        if nodes["pType"][i] == L.BVH:
            for c in (int(nodes["left"][i]), int(nodes["right"][i])):
                depth[c] = depth[i] + 1
                stack.append(c)
    tri = np.nonzero((depth >= 0) & (nodes["pType"] == L.TRIANGLE))[0]
    boxes = np.zeros(prim.nTri, dtype=L.bvh_dtype)
    if prim.nTri:
        check(lib.trq_bvh_build_nodes_triangles(verts.ctypes.data, prim.idxList.ctypes.data, prim.nTri, 0, boxes.ctypes.data), "leaves")
    nodes["mini"][tri] = boxes["mini"][nodes["pIndex"][tri]]
    nodes["maxi"][tri] = boxes["maxi"][nodes["pIndex"][tri]]
    inner = np.nonzero((depth >= 0) & (nodes["pType"] == L.BVH))[0]
    for i in inner[np.argsort(-depth[inner], kind="stable")]:
        l, r = nodes["left"][i], nodes["right"][i]
        nodes["mini"][i] = np.minimum(nodes["mini"][l], nodes["mini"][r])
        nodes["maxi"][i] = np.maximum(nodes["maxi"][l], nodes["maxi"][r])
    return Primitive(sphereList=prim.sphereList, squareList=prim.squareList, cubeList=prim.cubeList, triList=verts,
                     idxList=prim.idxList, bvhList=nodes)


def assert_records_match_reference(recs, want, hits=None, where=""):
    """Bit-exact comparison of HitRecord dumps on the rays the reference reports as hit. hits: the trq_hit rows of a GPU
    trace of the same rays; their sphere hits' uv comes from CUDA's atan2f / asinf, and is held to
    test_special_rays_cpu.assert_sphere_uv against the reference's shading normals instead."""
    assert np.array_equal(recs["hit"], want["hit"]), f"{where}: hit flags differ"
    m = want["hit"] == 1
    for k in ("t", "p", "gn", "sn", "front", "material"):
        assert np.array_equal(bits(recs[k][m]), bits(want[k][m])), f"{where}: {k} differs"
    if hits is None:
        assert np.array_equal(bits(recs["uv"][m]), bits(want["uv"][m])), f"{where}: uv differs"
    else:
        from .test_special_rays_cpu import assert_sphere_uv
        sph = m & (hits["pType"] == L.SPHERE)
        assert np.array_equal(bits(recs["uv"][m & ~sph]), bits(want["uv"][m & ~sph])), f"{where}: uv differs"
        if sph.any():
            assert_sphere_uv(recs["uv"][sph, 0], recs["uv"][sph, 1], want["gn"][sph], want["uv"][sph, 0], want["uv"][sph, 1],
                             f"{where}: sphere uv")
