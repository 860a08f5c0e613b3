"""Host restatement of trq_scene_update_primitives, shared by its tests (CPU and GPU)."""
import numpy as np

from tracer_b200 import layout as L
from tracer_b200.scene import Primitive


def primitive_leaves(records, p_type):
    """trq_bvh_build_node of every record (pIndex = its position): the leaf a scene update gives a leaf naming it."""
    from tracer_b200._lib import check, lib
    out = np.zeros(records.size, dtype=L.bvh_dtype)
    for k in range(records.size):
        lo, hi, m = (np.ascontiguousarray(records[f][k], dtype=np.float32) for f in ("box_mini", "box_maxi", "model"))
        check(lib.trq_bvh_build_node(lo.ctypes.data, hi.ctypes.data, m.ctypes.data, int(p_type), k, out[k:k + 1].ctypes.data),
              "trq_bvh_build_node")
    return out


def depths(bvh):
    """Depth of every node the root reaches, -1 elsewhere."""
    depth = np.full(bvh.size, -1, dtype=np.int64)
    depth[0] = 0
    stack = [0]
    while stack:
        i = stack.pop()
        if bvh["pType"][i] == L.BVH:
            for c in (int(bvh["left"][i]), int(bvh["right"][i])):
                depth[c] = depth[i] + 1
                stack.append(c)
    return depth


def update_on_host(prim, spheres=None, squares=None, cubes=None, verts=None):
    """trq_scene_update_primitives restated with numpy for a tree in any node numbering. Each list given replaces the
    primitive's. Reachable sphere / square / cube leaves of a replaced kind take mini / maxi of trq_bvh_build_node on their
    new record; triangle leaves follow `verts` as in util.refit_on_host; then the reachable interior nodes, deepest first,
    become the unions of their children with np.fmin / np.fmax (a NaN side is ignored, as by CUDA's fminf / fmaxf). Every
    other field and every node the root does not reach is kept. -> the updated Primitive."""
    from tracer_b200._lib import check, lib
    nodes = prim.bvhList.copy()
    depth = depths(nodes)
    reach = depth >= 0
    new = dict(sphereList=prim.sphereList, squareList=prim.squareList, cubeList=prim.cubeList, triList=prim.triList)
    for p_type, key, arr in ((L.SPHERE, "sphereList", spheres), (L.SQUARE, "squareList", squares), (L.CUBE, "cubeList", cubes)):
        if arr is None:
            continue
        arr = np.ascontiguousarray(arr)
        assert arr.dtype == new[key].dtype and arr.size == new[key].size, key
        new[key] = arr
        at = np.nonzero(reach & (nodes["pType"] == p_type))[0]
        if at.size:
            made = primitive_leaves(arr, p_type)
            nodes["mini"][at] = made["mini"][nodes["pIndex"][at]]
            nodes["maxi"][at] = made["maxi"][nodes["pIndex"][at]]
    if verts is not None:
        verts = np.ascontiguousarray(verts)
        assert verts.dtype == L.vertex_dtype and verts.size == prim.triList.size
        new["triList"] = verts
        at = np.nonzero(reach & (nodes["pType"] == L.TRIANGLE))[0]
        if at.size:
            made = np.zeros(prim.nTri, dtype=L.bvh_dtype)
            check(lib.trq_bvh_build_nodes_triangles(verts.ctypes.data, prim.idxList.ctypes.data, prim.nTri, 0, made.ctypes.data), "leaves")
            nodes["mini"][at] = made["mini"][nodes["pIndex"][at]]
            nodes["maxi"][at] = made["maxi"][nodes["pIndex"][at]]
    inner = np.nonzero(reach & (nodes["pType"] == L.BVH))[0]
    for i in inner[np.argsort(-depth[inner], kind="stable")]:
        l, r = nodes["left"][i], nodes["right"][i]
        nodes["mini"][i] = np.fmin(nodes["mini"][l], nodes["mini"][r])
        nodes["maxi"][i] = np.fmax(nodes["maxi"][l], nodes["maxi"][r])
    return Primitive(idxList=prim.idxList, bvhList=nodes, **new)
