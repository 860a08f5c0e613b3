"""Host restatement of trq_scene_rebuild, shared by the rebuild tests (CPU and GPU)."""
import ctypes as C

import numpy as np

from tracer_b200 import layout as L
from tracer_b200.scene import Primitive


def reachable(bvh):
    """Mask of the nodes the root reaches."""
    seen = np.zeros(bvh.size, dtype=bool)
    stack = [0]
    while stack:
        i = stack.pop()
        seen[i] = True
        if bvh["pType"][i] == L.BVH:
            stack += [int(bvh["left"][i]), int(bvh["right"][i])]
    return seen


def rebuild_on_host(prim, verts=None, gpu=None):
    """trq_scene_rebuild restated on the host: the leaves the root reaches, in bvhList order; triangle leaves made again
    from `verts` (None: the primitive's own) with trq_bvh_build_nodes_triangles, keeping pIndex; other leaves keep pType,
    pIndex and box with every other field zero; then trq_bvh_build_tree (gpu=None) or trq_bvh_build_tree_gpu on that
    list. Raises TrqError as the builder fails (TRQ_ERR_DEPTH). -> the rebuilt Primitive."""
    from tracer_b200._lib import check, lib
    verts = prim.triList if verts is None else np.ascontiguousarray(verts)
    old = prim.bvhList
    at = np.nonzero(reachable(old) & (old["pType"] != L.BVH))[0]
    n = at.size
    nodes = np.zeros(2 * n - 1, dtype=L.bvh_dtype)
    nodes["pType"][:n], nodes["pIndex"][:n] = old["pType"][at], old["pIndex"][at]
    nodes["mini"][:n], nodes["maxi"][:n] = old["mini"][at], old["maxi"][at]
    tri = np.nonzero(nodes["pType"][:n] == L.TRIANGLE)[0]
    if tri.size:
        # one call for all of them: leaf k of the call is trq_bvh_build_node of triangle idx[k], pIndex = pIndexBase + k
        p = nodes["pIndex"][tri]
        idx = np.ascontiguousarray(prim.idxList.reshape(-1, 3)[p])
        made = np.zeros(tri.size, dtype=L.bvh_dtype)
        check(lib.trq_bvh_build_nodes_triangles(verts.ctypes.data, idx.ctypes.data, tri.size, 0, made.ctypes.data), "leaves")
        made["pIndex"] = p
        nodes[tri] = made
    if n > 1:
        nn, depth = C.c_uint32(0), C.c_uint32(0)
        if gpu is None:
            check(lib.trq_bvh_build_tree(nodes.ctypes.data, n, C.byref(nn), C.byref(depth)), "trq_bvh_build_tree")
        else:
            check(lib.trq_bvh_build_tree_gpu(nodes.ctypes.data, n, int(gpu), C.byref(nn), C.byref(depth)), "trq_bvh_build_tree_gpu")
    return Primitive(sphereList=prim.sphereList, squareList=prim.squareList, cubeList=prim.cubeList, triList=verts,
                     idxList=prim.idxList, bvhList=nodes)
