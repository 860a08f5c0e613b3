"""The Morton-order builder's rules (include/tracer_rq.h, kernels/morton_build.cuh) written again with numpy, a structural
check for its trees, the host restatement's entry point and the leaf sets the Morton tests share (CPU and GPU)."""
import ctypes as C

import numpy as np

from tracer_b200 import harness as H, layout as L

F = np.float32
QMAX = (1 << 21) - 1


def quantise_axis(v):
    """q of every centroid component on one axis (float32 arithmetic, one rounding per operation)."""
    v = np.asarray(v, dtype=F)
    q = np.zeros(v.size, dtype=np.uint64)
    fin = np.isfinite(v)
    if fin.any():
        lo, hi = v[fin].min(), v[fin].max()
        with np.errstate(over="ignore", invalid="ignore"):
            ext = F(hi - lo)
        if np.isfinite(ext) and ext > 0:
            t = np.floor(((v[fin] - lo) / ext) * F(1 << 21))
            assert t.dtype == F and (t >= 0).all()
            q[fin] = np.minimum(t, F(QMAX)).astype(np.uint64)
    q[np.isnan(v) | (v == np.inf)] = QMAX
    return q


def morton_codes(leaves):
    with np.errstate(over="ignore", invalid="ignore"):
        c = leaves["mini"] + (leaves["maxi"] - leaves["mini"]) / F(2)
    code = np.zeros(leaves.size, dtype=np.uint64)
    for axis, shift in ((0, 2), (1, 1), (2, 0)):
        q = quantise_axis(c[:, axis])
        for i in range(21):
            code |= ((q >> np.uint64(i)) & np.uint64(1)) << np.uint64(3 * i + shift)
    return code


def box_min(a, b):
    """CUDA's fminf: NaN ignored, -0.0 below +0.0."""
    zero = (a == 0) & (b == 0)
    return np.where(zero, np.where(np.signbit(a), a, b), np.fmin(a, b))


def box_max(a, b):
    """CUDA's fmaxf: NaN ignored, +0.0 above -0.0."""
    zero = (a == 0) & (b == 0)
    return np.where(zero, np.where(np.signbit(a), b, a), np.fmax(a, b))


def morton_tree(leaves, clamp=True):
    """-> (nodes, maxDepth, sorted order). clamp=False: the Karras tree without the depth clamp (numbering as with it)."""
    n = leaves.size
    nodes = np.zeros(2 * n - 1, dtype=L.bvh_dtype)
    if n == 1:
        nodes[0] = leaves[0]
        nodes["parent"][0] = 0
        return nodes, 0, np.zeros(1, dtype=np.int64)
    code = morton_codes(leaves)
    order = np.argsort(code, kind="stable")
    sc = [int(x) for x in code[order]]

    def split(a, b, d):
        m = b - a + 1
        if sc[a] == sc[b]:
            s, axis = m // 2, 0
        else:
            h = (sc[a] ^ sc[b]).bit_length() - 1
            axis = 2 - h % 3
            s = next(p for p in range(a + 1, b + 1) if (sc[p] >> h) & 1) - a
        if clamp:
            lim = 1 << (31 - d)
            s = min(max(s, m - lim, 1), lim, m - 1)
        return s, axis

    nodes[1:n + 1] = leaves
    s, axis = split(0, n - 1, 0)
    g_root = s - 1
    index = lambda g: n + 1 + g if g < g_root else n + g        # noqa: E731
    stack = [(0, n - 1, 0, 0, 0, s, axis)]                       # a, b, depth, self, parent, left size, axis
    post = []
    max_depth = 0
    while stack:
        a, b, d, me, parent, s, axis = stack.pop()
        max_depth = max(max_depth, d)
        kids = []
        for lo, hi in ((a, a + s - 1), (a + s, b)):
            if lo == hi:
                kid = 1 + int(order[lo])
                nodes["parent"][kid] = me
            else:
                cs, caxis = split(lo, hi, d + 1)
                kid = index(lo + cs - 1)
                stack.append((lo, hi, d + 1, kid, me, cs, caxis))
            kids.append(kid)
        nodes[me]["parent"], nodes[me]["left"], nodes[me]["right"] = parent, kids[0], kids[1]
        nodes[me]["axis"], nodes[me]["pType"] = axis, L.BVH
        post.append((d, me))
    for _, me in sorted(post, reverse=True):                     # deepest first: children before parents
        l, r = nodes["left"][me], nodes["right"][me]
        nodes["mini"][me] = box_min(nodes["mini"][l], nodes["mini"][r])
        nodes["maxi"][me] = box_max(nodes["maxi"][l], nodes["maxi"][r])
    return nodes, max_depth, order


def host_morton(leaves):
    """trq_bvh_build_tree_morton -> (status, nNode, maxDepth, nodes)."""
    from tracer_b200._lib import lib
    n = leaves.size
    nodes = np.zeros(2 * n - 1, dtype=L.bvh_dtype)
    nodes[:n] = leaves
    nn, d = C.c_uint32(0xdead), C.c_uint32(0xdead)
    rc = lib.trq_bvh_build_tree_morton(nodes.ctypes.data, n, C.byref(nn), C.byref(d))
    return rc, nn.value, d.value, nodes


def check_morton_structure(bvh, leaves, order):
    """Every leaf once, at 1..n in list order; parent links agree; interiors at the gap numbering; boxes are unions.
    -> deepest interior level."""
    n = leaves.size
    assert bvh.size == 2 * n - 1
    if n == 1:
        assert bvh[0].tobytes() == leaves[0].tobytes() or (bvh["parent"][0] == 0)
        return 0
    lv = bvh[1:n + 1].copy()
    lv["parent"] = leaves["parent"]
    assert lv.tobytes() == leaves.tobytes(), "leaves at 1..n in list order, every field but parent kept"
    inter = np.concatenate([[0], np.arange(n + 1, bvh.size)])
    assert (bvh["pType"][inter] == L.BVH).all() and bvh["parent"][0] == 0
    assert (bvh["pIndex"][inter] == 0).all() and (bvh["pad"][inter] == 0).all()
    assert (bvh["pad0"][inter] == 0).all() and (bvh["pad1"][inter] == 0).all()
    l, r = bvh["left"][inter], bvh["right"][inter]
    assert np.array_equal(bvh["parent"][l], inter) and np.array_equal(bvh["parent"][r], inter)
    assert np.array_equal(np.sort(np.concatenate([l, r])), np.arange(1, bvh.size)), "every non-root node a child once"
    assert np.array_equal(bvh["mini"][inter], np.fmin(bvh["mini"][l], bvh["mini"][r]))
    assert np.array_equal(bvh["maxi"][inter], np.fmax(bvh["maxi"][l], bvh["maxi"][r]))
    # sorted span of every node, depth, and the gap numbering
    pos = np.empty(n, dtype=np.int64)
    pos[order] = np.arange(n)
    lo, hi, depth = {}, {}, {0: 0}
    stack, walk = [0], []
    while stack:
        i = stack.pop()
        walk.append(i)
        if bvh["pType"][i] == L.BVH:
            for c in (int(bvh["left"][i]), int(bvh["right"][i])):
                depth[c] = depth[i] + 1
                stack.append(c)
    for i in reversed(walk):
        if bvh["pType"][i] == L.BVH:
            a, b = int(bvh["left"][i]), int(bvh["right"][i])
            lo[i], hi[i] = lo[a], hi[b]
            assert hi[a] + 1 == lo[b], "children are adjacent sorted spans"
        else:
            lo[i] = hi[i] = int(pos[i - 1])
    g_root = hi[int(bvh["left"][0])]
    for i in inter[1:]:
        g = hi[int(bvh["left"][i])]
        assert i == (n + 1 + g if g < g_root else n + g), f"node {i} splits gap {g}"
    return max(depth[i] for i in inter)


# ---------------------------------------------------------------------------------------------------------- leaf sets
def point_leaves(points, p_type=L.TRIANGLE):
    p = np.asarray(points, dtype=F)
    lv = np.zeros(p.shape[0], dtype=L.bvh_dtype)
    lv["pType"], lv["pIndex"] = p_type, np.arange(p.shape[0])
    lv["mini"], lv["maxi"] = p, p
    return lv


def chain_points(copies=1):
    """63 centroids each quantising to one bit of the code (x, y, z at 2^(i-21), i = 0..20) and one at (1, 1, 1) that
    sets every bit: 64 codes that Karras' rule splits one leaf at a time, a chain 60+ levels deep without the clamp.
    Each point `copies` times (a power of two keeps the leaf count 2^k)."""
    pts = [[1.0, 1.0, 1.0]]
    for axis in range(3):
        for i in range(21):
            p = [0.0, 0.0, 0.0]
            p[axis] = 2.0 ** (i - 21)
            pts.append(p)
    return np.repeat(np.array(pts), copies, axis=0)


def mixed_leaves(seed, n=400):
    """Sphere, square, cube and triangle leaves from test_gpu_tree_shapes' generator, in one list."""
    from .test_gpu_tree_shapes import Leaves, mixed
    lv = Leaves()
    mixed(np.random.default_rng(seed), lv, n)
    out = np.zeros(len(lv.items), dtype=L.bvh_dtype)
    for k, (t, p, lo, hi) in enumerate(lv.items):
        out[k]["pType"], out[k]["pIndex"], out[k]["mini"], out[k]["maxi"] = t, p, lo, hi
    return lv, out


def reference_cornell_leaves():
    prim = H.scene_reference_cornell()
    n = (prim.bvhList.size + 1) // 2
    lv = prim.bvhList[1:n + 1].copy()
    lv["parent"] = 0
    return prim, lv


def rebuild_leaves(prim, verts=None):
    """The leaf list of trq_scene_rebuild (include/tracer_rq.h): the leaves the root reaches in bvhList order, triangle
    leaves made again from `verts` keeping pIndex, the others keeping pType, pIndex and box, every other field zero."""
    from tracer_b200._lib import check, lib
    verts = prim.triList if verts is None else np.ascontiguousarray(verts)
    old = prim.bvhList
    reach = np.zeros(old.size, dtype=bool)
    stack = [0]
    while stack:
        i = stack.pop()
        reach[i] = True
        if old["pType"][i] == L.BVH:
            stack += [int(old["left"][i]), int(old["right"][i])]
    at = np.nonzero(reach & (old["pType"] != L.BVH))[0]
    lv = np.zeros(at.size, dtype=L.bvh_dtype)
    for f in ("pType", "pIndex", "mini", "maxi"):
        lv[f] = old[f][at]
    tri = np.nonzero(lv["pType"] == L.TRIANGLE)[0]
    if tri.size:
        idx = np.ascontiguousarray(prim.idxList.reshape(-1, 3)[lv["pIndex"][tri]])
        made = np.zeros(tri.size, dtype=L.bvh_dtype)
        check(lib.trq_bvh_build_nodes_triangles(verts.ctypes.data, idx.ctypes.data, tri.size, 0, made.ctypes.data), "leaves")
        made["pIndex"] = lv["pIndex"][tri]
        lv[tri] = made
    return lv


def morton_rebuild_on_host(prim, verts=None):
    """trq_scene_rebuild with TRQ_BUILD_MORTON restated: the Morton host restatement over rebuild_leaves. -> Primitive."""
    from tracer_b200.scene import Primitive
    verts = prim.triList if verts is None else np.ascontiguousarray(verts)
    rc, _, _, nodes = host_morton(rebuild_leaves(prim, verts))
    assert rc == 0
    return Primitive(sphereList=prim.sphereList, squareList=prim.squareList, cubeList=prim.cubeList, triList=verts,
                     idxList=prim.idxList, bvhList=nodes)
