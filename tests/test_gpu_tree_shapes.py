"""Caller-built trees against the oracle.

trq_scene_create / trq_scene_create_device accept any tree in the reference layout (include/tracer_rq.h): interior depth
up to 31, any node numbering with the root at 0 (BVH.hh:264), leaves of any pType, boxes that need not contain their
children, and -- for trq_scene_create only -- nodes the root does not reach. The trees here are built by hand, not by
BVHBuilder, so that the host walk and the device plan kernels number something other than the builder's post-order, the
far-child stack is filled to its exact bound (32 pending far children at depth 31), and the refit runs on trees whose
numbering and unreachable nodes it cannot assume away. Every answer is compared with port.trace, the strict-IEEE
restatement of Scene::hit (Render.hh:132-252).

The depth-boundary tests at the top need no GPU.
"""
import ctypes as C

import numpy as np
import pytest

from tracer_b200 import harness as H, layout as L
from tracer_b200._lib import ERR_DEPTH, ERR_NO_DEVICE, OK, lib
from tracer_b200.scene import Primitive

from .util import refit_on_host

f32 = np.float32
MAX_DEPTH = 31                         # deepest interior level the reference's 32-bit trail represents (Render.hh:140)
TOP_MAX = 2047                         # interior nodes numbered breadth-first at the front of the packed array
COLD_WORDS = 9                         # per-ray shared-memory words beside the far-child stack (trace_kernels.cuh)
SMEM_PER_SM, SMEM_DYNAMIC_MAX, SMEM_BLOCK_RESERVE = 228 * 1024, 226 * 1024, 1024


# ---------------------------------------------------------------------------------------------------------------- leaves
class Leaves:
    """Leaf payloads and the primitive arrays they index. items[k] = (pType, pIndex, box_lo, box_hi)."""

    def __init__(self):
        self.tri, self.spheres, self.squares, self.cubes, self.items = [], [], [], [], []

    def triangle(self, p):
        p = np.asarray(p, dtype=f32).reshape(3, 3)
        self.items.append((L.TRIANGLE, len(self.tri), p.min(0), p.max(0)))
        self.tri.append(p)

    def sphere(self, r, c):
        s = H.make_sphere(r, c, 7)
        self.items.append((L.SPHERE, len(self.spheres), s["box_mini"].copy(), s["box_maxi"].copy()))
        self.spheres.append(s)

    def square(self, axis_i, range_i, axis_j, range_j, axis_k, k):
        s = H.make_square(axis_i, range_i, axis_j, range_j, axis_k, k, 4)
        self.items.append((L.SQUARE, len(self.squares), s["box_mini"].copy(), s["box_maxi"].copy()))
        self.squares.append(s)

    def cube(self, model):
        c = H.make_cube(model, 19)
        node = np.zeros(1, dtype=L.bvh_dtype)                 # BVH::buildNode: world box of the 8 transformed corners
        lo, hi = np.zeros(3, dtype=f32), np.ones(3, dtype=f32)
        m = np.ascontiguousarray(c["model"], dtype=f32)
        lib.trq_bvh_build_node(lo.ctypes.data, hi.ctypes.data, m.ctypes.data, L.CUBE, len(self.cubes), node.ctypes.data)
        self.items.append((L.CUBE, len(self.cubes), node["mini"][0].copy(), node["maxi"][0].copy()))
        self.cubes.append(c)

    def other(self, p_type, p_index, lo, hi):
        """A leaf the reference dispatches to `default: break` (Render.hh:241): never hit."""
        self.items.append((p_type, p_index, np.asarray(lo, dtype=f32), np.asarray(hi, dtype=f32)))

    def repeat(self, k):
        """A second leaf naming the same primitive as leaf k."""
        self.items.append(self.items[k])

    def arrays(self):
        out = {}
        if self.tri:
            pos = np.concatenate(self.tri)
            idx = np.arange(pos.shape[0], dtype=np.uint32)
            out["triList"], out["idxList"] = H.make_vertices(pos, idx.reshape(-1, 3)), idx
        for k, v, dt in (("sphereList", self.spheres, L.sphere_dtype), ("squareList", self.squares, L.square_dtype),
                         ("cubeList", self.cubes, L.cube_dtype)):
            if v:
                out[k] = np.array(v, dtype=dt)
        return out


def soup(rng, lv, n, extent=0.15):
    for _ in range(n):
        c = rng.uniform(0, 1, 3)
        lv.triangle(c + rng.uniform(-extent, extent, (3, 3)))


def lattice(rng, lv, n):
    """Integer-lattice triangles: exact ties, duplicates, zero-area triangles, flat boxes (test_gpu_fuzz.scenes)."""
    pts = rng.integers(-3, 4, (n, 3, 3)).astype(f32)
    pts[::9, 2] = pts[::9, 1]
    pts[1::13] = pts[0::13][: len(pts[1::13])]
    for p in pts:
        lv.triangle(p)


def mixed(rng, lv, n):
    for k in range(n):
        c = rng.uniform(-3, 3, 3).astype(f32)
        kind = k % 4
        if kind == 0:
            lv.sphere(float(rng.uniform(0.1, 0.6)), c)
        elif kind == 1:
            a, b = sorted(rng.uniform(-3, 3, 2)), sorted(rng.uniform(-3, 3, 2))
            lv.square(0, (f32(a[0]), f32(a[1])), 2, (f32(b[0]), f32(b[1])), 1, f32(c[1]))
        elif kind == 2:
            m = H.translation4x4(*c) @ H.rotation4x4(float(rng.uniform(0, 3)), (0, 1, 0)) @ H.scale4x4(*rng.uniform(0.1, 0.8, 3))
            lv.cube(m)
        else:
            lv.triangle(c + rng.uniform(-0.5, 0.5, (3, 3)))


# ------------------------------------------------------------------------------------------------------------- topology
class Topo:
    """A binary tree before numbering: left[i] / right[i] (-1 at a leaf), leaf[i] = index into Leaves.items (-1 at an
    interior node)."""

    def __init__(self):
        self.left, self.right, self.leaf = [], [], []
        self.root = -1

    def add(self, left=-1, right=-1, leaf=-1):
        self.left.append(left); self.right.append(right); self.leaf.append(leaf)
        return len(self.leaf) - 1

    def depths(self):
        d = np.full(len(self.leaf), -1, dtype=np.int64)
        d[self.root] = 0
        stack = [self.root]
        while stack:
            i = stack.pop()
            if self.leaf[i] < 0:
                for c in (self.left[i], self.right[i]):
                    d[c] = d[i] + 1
                    stack.append(c)
        return d

    def max_interior_depth(self):
        d = self.depths()
        inner = np.array(self.leaf) < 0
        return int(d[inner].max()) if inner.any() else 0


def split_tree(rng, topo, leaves, balanced=False):
    """Recursive split of the leaf list at a uniform random point (balanced: within the middle half)."""
    if len(leaves) == 1:
        return topo.add(leaf=leaves[0])
    m = len(leaves)
    k = int(rng.integers(max(1, m // 4), max(2, 3 * m // 4 + 1))) if balanced else int(rng.integers(1, m))
    a = split_tree(rng, topo, leaves[:k], balanced)
    b = split_tree(rng, topo, leaves[k:], balanced)
    return topo.add(a, b)


def random_split(rng, n_leaves, balanced=False):
    for _ in range(100):
        t = Topo()
        t.root = split_tree(rng, t, list(range(n_leaves)), balanced)
        if t.max_interior_depth() <= MAX_DEPTH:
            return t
    raise AssertionError("no random split within the depth limit")


def comb(depth, interior_left):
    """Interior nodes at depths 0..depth, each with one leaf child and one interior child (the deepest: two leaves). Leaf k
    hangs at depth k + 1; leaf depth + 1 is the deepest one's second child."""
    t = Topo()
    node = t.add(leaf=depth + 1)
    for k in range(depth, -1, -1):
        leaf = t.add(leaf=k)
        node = t.add(node, leaf) if interior_left else t.add(leaf, node)
    t.root = node
    return t


def spine(rng, sizes):
    """A depth-31 spine; spine node d carries a bushy random subtree of sizes[d] leaves as its other child."""
    assert len(sizes) == MAX_DEPTH + 1
    t = Topo()
    first = 0
    subs = []
    for d, m in enumerate(sizes):
        for _ in range(100):
            mark = len(t.leaf)
            r = split_tree(rng, t, list(range(first, first + m)), balanced=True)
            t.root = r
            sub_d = t.max_interior_depth() if m > 1 else -1
            if d + 1 + sub_d <= MAX_DEPTH:
                break
            del t.left[mark:], t.right[mark:], t.leaf[mark:]
        else:
            raise AssertionError("no subtree within the depth limit")
        subs.append(r)
        first += m
    node = t.add(leaf=first)                                   # the spine ends in two leaves at depth 32
    node = t.add(subs[-1], node) if rng.random() < 0.5 else t.add(node, subs[-1])
    for d in range(MAX_DEPTH - 1, -1, -1):
        node = t.add(node, subs[d]) if rng.random() < 0.5 else t.add(subs[d], node)
    t.root = node
    return t, first + 1


# ------------------------------------------------------------------------------------------------------------ numbering
def numbering(topo, how, rng):
    """-> perm[topology node] = index in bvhList, root at 0.
    post: the builder's order (leaves 1..N left to right, interior nodes after them in post-order);
    bfs: breadth-first; random: a random permutation of 1..n-1, with left / right swapped at random first."""
    n = len(topo.leaf)
    perm = np.zeros(n, dtype=np.int64)
    if how == "random":
        for i in range(n):
            if topo.leaf[i] < 0 and rng.random() < 0.5:
                topo.left[i], topo.right[i] = topo.right[i], topo.left[i]
        others = [i for i in range(n) if i != topo.root]
        perm[others] = rng.permutation(n - 1) + 1
        return perm
    order = []
    if how == "bfs":
        q = [topo.root]
        for i in q:
            order.append(i)
            if topo.leaf[i] < 0:
                q += [topo.left[i], topo.right[i]]
    else:
        leaves, post = [], []

        def walk(i):
            if topo.leaf[i] >= 0:
                leaves.append(i)
                return
            walk(topo.left[i]); walk(topo.right[i])
            post.append(i)
        walk(topo.root)
        order = [topo.root] + leaves + [i for i in post if i != topo.root]
    perm[order] = np.arange(n)
    return perm


# ---------------------------------------------------------------------------------------------------------------- boxes
def tight_boxes(topo, lv):
    n = len(topo.leaf)
    lo, hi = np.zeros((n, 3), dtype=f32), np.zeros((n, 3), dtype=f32)
    d = topo.depths()
    for i in np.argsort(-d, kind="stable"):
        if topo.leaf[i] >= 0:
            _, _, lo[i], hi[i] = lv.items[topo.leaf[i]]
        else:
            lo[i] = np.minimum(lo[topo.left[i]], lo[topo.right[i]])
            hi[i] = np.maximum(hi[topo.left[i]], hi[topo.right[i]])
    return lo, hi


def boxes(topo, lv, how, rng):
    """tight: unions of the children; inflated: every box grown by a random margin, bottom-up (still nesting);
    nonnest: random boxes that overlap their subtree's geometry but need not contain their children;
    inf: inflated, and a few non-root boxes with an infinite extent."""
    lo, hi = tight_boxes(topo, lv)
    if how == "tight":
        return lo, hi
    ext = f32(np.max(hi[topo.root] - lo[topo.root]))
    if how in ("inflated", "inf"):
        d = topo.depths()
        for i in np.argsort(-d, kind="stable"):
            if topo.leaf[i] < 0:
                lo[i] = np.minimum(lo[topo.left[i]], lo[topo.right[i]])
                hi[i] = np.maximum(hi[topo.left[i]], hi[topo.right[i]])
            lo[i] -= (rng.random(3) * 0.05 * ext).astype(f32)
            hi[i] += (rng.random(3) * 0.05 * ext).astype(f32)
        if how == "inf":
            for i in rng.choice([j for j in range(len(topo.leaf)) if j != topo.root], 12, replace=False):
                ax = int(rng.integers(3))
                if rng.random() < 0.5:
                    lo[i, ax] = -np.inf
                else:
                    hi[i, ax] = np.inf
        return lo, hi
    assert how == "nonnest"
    size = hi - lo
    a = (rng.uniform(-0.15, 0.3, lo.shape) * size).astype(f32)
    b = (rng.uniform(-0.15, 0.3, lo.shape) * size).astype(f32)
    return lo + a, hi - b


def make_prim(topo, lv, perm, lo, hi):
    n = len(topo.leaf)
    bvh = np.zeros(n, dtype=L.bvh_dtype)
    for i in range(n):
        j = perm[i]
        if topo.leaf[i] >= 0:
            p_type, p_index, _, _ = lv.items[topo.leaf[i]]
            bvh["pType"][j], bvh["pIndex"][j] = p_type, p_index
        else:
            bvh["pType"][j] = L.BVH
            bvh["left"][j], bvh["right"][j] = perm[topo.left[i]], perm[topo.right[i]]
            bvh["parent"][perm[topo.left[i]]] = bvh["parent"][perm[topo.right[i]]] = j
        bvh["mini"][j], bvh["maxi"][j] = lo[i], hi[i]
    return Primitive(bvhList=bvh, **lv.arrays())


def comb_leaves(depth, interior_left, tie, kind="triangle"):
    """Leaf k at x = 100 - k: every leaf is further along +x than every leaf below it, so a +x ray hits both children at
    every level and the interior child is nearer -- depth + 1 far children are pending at the deepest node. tie: every
    leaf box starts at x = 50, so both children tie on entry t at every level ("ties go right", Render.hh:174)."""
    lv = Leaves()
    for k in range(depth + 2):
        x = f32(100 - k)
        if kind == "square":
            lv.square(1, (-1, 1), 2, (-1, 1), 0, x)
        else:
            lv.triangle([[x, -1, -1], [x, 3, -1], [x, -1, 3]])
    if tie:
        lv.items = [(t, p, np.array([50, lo[1], lo[2]], dtype=f32), hi) for t, p, lo, hi in lv.items]
    return lv


def comb_prim(depth, interior_left=True, tie=False, how="post", kind="triangle", seed=0):
    topo = comb(depth, interior_left)
    lv = comb_leaves(depth, interior_left, tie, kind)
    perm = numbering(topo, how, np.random.default_rng(seed))
    lo, hi = boxes(topo, lv, "tight", None)
    return make_prim(topo, lv, perm, lo, hi), topo, lv


# ------------------------------------------------------------------------------------------------------- the tree cases
def tree_case(name):
    """-> (Primitive, Topo, Leaves). Every case is seeded by its name."""
    rng = np.random.default_rng(sum(map(ord, name)))
    lv = Leaves()
    shape, how, box = name.split("-")[:3]
    if shape.startswith("comb"):                               # comb<L|R><near|tie>[sq]
        prim, topo, lv = comb_prim(MAX_DEPTH, interior_left=shape[4] == "L", tie="tie" in shape, how=how,
                                   kind="square" if shape.endswith("sq") else "triangle", seed=int(rng.integers(1 << 30)))
        return prim, topo, lv
    if shape == "spine":
        sizes = [64] * 16 + [8] * 8 + [4] * 4 + [2] * 3 + [1]
        topo, n = spine(rng, sizes)
        soup(rng, lv, n, 0.05)
    elif shape in ("top2047", "top2048"):
        n = 2048 if shape == "top2047" else 2049
        soup(rng, lv, n, 0.02)
        topo = random_split(rng, n, balanced=True)
    else:
        leaves = name.split("-")[3]
        if leaves == "soup":
            soup(rng, lv, 300)
        elif leaves == "lattice":
            lattice(rng, lv, 300)
        elif leaves == "mixed":
            mixed(rng, lv, 160)
        elif leaves == "odd":                                  # unknown pTypes and repeated primitives among mixed leaves
            mixed(rng, lv, 120)
            for k in range(6):
                lv.other(L.UNKNOW if k % 2 else 9, k, rng.uniform(-3, 0, 3), rng.uniform(0, 3, 3))
            for k in range(0, 120, 7):
                lv.repeat(k)
        topo = random_split(rng, len(lv.items))
    perm = numbering(topo, how, rng)
    lo, hi = boxes(topo, lv, box, rng)
    return make_prim(topo, lv, perm, lo, hi), topo, lv


TREES = ["split-post-tight-soup", "split-bfs-inflated-mixed", "split-random-nonnest-lattice", "split-random-inf-odd",
         "split-bfs-nonnest-mixed",
         "combLnear-post-tight", "combRnear-random-tight", "combLtie-random-tight", "combRtie-bfs-tight",
         "combLnearsq-bfs-tight",
         "spine-random-tight", "top2047-bfs-tight", "top2048-random-inflated"]


# ------------------------------------------------------------------------------------------------------------------ rays
def geometry_bounds(lv):
    lo = np.min([it[2] for it in lv.items if np.isfinite(it[2]).all()], axis=0)
    hi = np.max([it[3] for it in lv.items if np.isfinite(it[3]).all()], axis=0)
    return lo.astype(f32), hi.astype(f32)


def _normalized(rays):
    lib.trqh_normalize_rays(rays.ctypes.data, rays.size)
    bad = ~np.isfinite(rays["d"]).all(axis=1)
    rays["d"][bad] = np.array([0, 0, 1], dtype=f32)
    return rays


def aimed_rays(rng, targets, lo, hi):
    """One ray per target point, from a random point outside the scene's bounds."""
    c, diag = (lo + hi) * f32(0.5), f32(np.linalg.norm(hi - lo)) + f32(1)
    rays = np.zeros(len(targets), dtype=L.ray_dtype)
    u = rng.normal(size=(len(targets), 3))
    rays["o"] = (c + diag * u / np.linalg.norm(u, axis=1, keepdims=True)).astype(f32)
    rays["d"] = (np.asarray(targets, dtype=f32) - rays["o"]).astype(f32)
    rays["tmax"] = L.FLT_MAX
    return _normalized(rays)


def tree_rays(rng, prim, lv, n=3000):
    """Rays aimed at every leaf's primitive, camera rays, adversarial rays (test_gpu_fuzz) and random rays."""
    from .test_gpu_fuzz import adversarial_rays
    lo, hi = geometry_bounds(lv)
    targets = [blo + (bhi - blo) * rng.uniform(0.2, 0.8, 3).astype(f32) for _, _, blo, bhi in lv.items]
    c, diag = (lo + hi) * f32(0.5), f32(np.linalg.norm(hi - lo))
    parts = [aimed_rays(rng, targets, lo, hi),
             H.camera_rays(c + np.array([0.3, 0.5, -2.5], dtype=f32) * diag, c, f32(0.8), 48, 32),
             H.random_rays(n, seed=int(rng.integers(1 << 30)), lo=lo - 0.2 * diag, hi=hi + 0.2 * diag)]
    adv = adversarial_rays(rng, Primitive(**{**prim.__dict__, "bvhList": _finite_root(prim.bvhList)}), n)
    bad = ~np.isfinite(adv["o"]).all(axis=1)                   # origins put on an infinite box plane
    adv["o"][bad] = c
    parts.append(adv)
    return np.ascontiguousarray(np.concatenate(parts))


def _finite_root(bvh):
    b = bvh.copy()
    b["mini"] = np.where(np.isfinite(b["mini"]), b["mini"], 0)
    b["maxi"] = np.where(np.isfinite(b["maxi"]), b["maxi"], 1)
    return b


def comb_rays(rng, lv, n=500):
    """+x rays through every leaf of a comb (from x = 0, inside the y / z extent of all leaves) and their -x mirror."""
    rays = np.zeros(2 * n, dtype=L.ray_dtype)
    rays["o"][:n, 1:] = rng.uniform(-0.9, 0.9, (n, 2)).astype(f32)
    rays["d"][:n, 0] = 1
    rays["o"][n:, 0] = 200
    rays["o"][n:, 1:] = rays["o"][:n, 1:]
    rays["d"][n:, 0] = -1
    rays["tmax"] = L.FLT_MAX
    return rays


def with_finite_tmax(rng, rays, lv):
    lo, hi = geometry_bounds(lv)
    r = rays.copy()
    r["tmax"] = (rng.uniform(0.05, 1.5, r.size) * np.linalg.norm(hi - lo)).astype(f32)
    return r


# ------------------------------------------------------------------------------------------------------ expected values
def expected_info(prim):
    """nInterior, nLeaf, maxDepth of the part of bvhList the root reaches, computed with numpy."""
    b = prim.bvhList
    depth = np.full(b.size, -1, dtype=np.int64)
    depth[0] = 0
    stack = [0]
    while stack:
        i = stack.pop()
        if b["pType"][i] == L.BVH:
            for ch in (int(b["left"][i]), int(b["right"][i])):
                depth[ch] = depth[i] + 1
                stack.append(ch)
    reach = depth >= 0
    inner = reach & (b["pType"] == L.BVH)
    n_inner = int(inner.sum())
    return dict(nNode=b.size, nInterior=n_inner, nLeaf=int((reach & ~inner).sum()),
                maxDepth=int(depth[inner].max()) if n_inner else 0, topNodes=min(TOP_MAX, n_inner),
                nTri=int((reach & (b["pType"] == L.TRIANGLE)).sum()), nSphere=int((reach & (b["pType"] == L.SPHERE)).sum()))


def expected_staging(name, max_depth, top_nodes):
    """(usable, staged nodes) of launch configuration `name` ("<block>x<CTAs per SM> top=<bool>") for a tree of this
    depth: per-CTA shared memory = far-child stack (maxDepth + 1 entries) + cold words per ray + staged nodes."""
    block, rest = name.split("x", 1)
    block, minb, top = int(block), int(rest.split()[0]), rest.endswith("true")
    per_ray = (max_depth + 1 + COLD_WORDS) * block * 4
    budget = min(SMEM_PER_SM // minb - SMEM_BLOCK_RESERVE, SMEM_DYNAMIC_MAX)
    staged = min((budget - per_ray) // 64, top_nodes) if top and budget > per_ray else 0
    return per_ray + staged * 64 <= SMEM_DYNAMIC_MAX and not (top and staged == 0), staged


# --------------------------------------------------------------------------------------------------- the depth boundary
def _create(prim):
    h = C.c_void_p(None)
    d = prim.desc()
    rc = lib.trq_scene_create(C.byref(d), 0, C.byref(h))
    if h.value:
        lib.trq_scene_destroy(h)
    return rc


@pytest.mark.parametrize("interior_left", [True, False])
def test_interior_depth_31_is_accepted_and_32_refused(built, interior_left):
    """The host walk accepts a comb whose deepest interior node is at depth 31 and refuses depth 32 (the 32-bit trail of
    Render.hh:140). Without a device an accepted tree gets TRQ_ERR_NO_DEVICE: validation runs first, on the host."""
    deep, _, _ = comb_prim(MAX_DEPTH, interior_left)
    assert expected_info(deep)["maxDepth"] == 31
    rc = _create(deep)
    assert rc == (OK if lib.trq_device_count() > 0 else ERR_NO_DEVICE), lib.trq_last_error_string()
    too_deep, _, _ = comb_prim(MAX_DEPTH + 1, interior_left)
    assert _create(too_deep) == ERR_DEPTH and b"trail" in lib.trq_last_error_string()


def test_generated_trees_are_what_they_claim(built):
    """The generators themselves: consistent links, the depths and sizes each case is meant to have."""
    for name in TREES:
        prim, topo, lv = tree_case(name)
        b = prim.bvhList
        inner = np.nonzero(b["pType"] == L.BVH)[0]
        assert b["parent"][0] == 0
        for i in inner:
            assert b["parent"][b["left"][i]] == i and b["parent"][b["right"][i]] == i and b["left"][i] != b["right"][i]
        e = expected_info(prim)
        assert e["nInterior"] + e["nLeaf"] == b.size and e["nLeaf"] == len(lv.items), name
        assert e["maxDepth"] <= MAX_DEPTH, name
        if name.startswith(("comb", "spine")):
            assert e["maxDepth"] == MAX_DEPTH, name
        if name.startswith("spine"):                           # more interior nodes than configuration 1 stages at depth 31
            assert e["nInterior"] > expected_staging("1024x1 top=true", MAX_DEPTH, TOP_MAX)[1]
        if name.startswith("top"):
            assert e["nInterior"] == int(name[3:7]), name
        if name.endswith("odd"):
            assert {L.UNKNOW, 9} <= set(b["pType"].tolist())
            leaves = b[b["pType"] != L.BVH]
            keys = list(zip(leaves["pType"].tolist(), leaves["pIndex"].tolist()))
            assert len(set(keys)) < len(keys)
        if name.startswith(("combLnear", "combRnear")):        # the leaves are ordered along +x as the stack bound needs
            leaf_x = b["mini"][b["pType"] != L.BVH][:, 0]
            assert np.unique(leaf_x).size == MAX_DEPTH + 2


# -------------------------------------------------------------------------------------------------------- GPU: parity
def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _check_configurations(scene, name):
    """Every configuration the shared-memory formula says fits must be offered, with the staged count it predicts; at
    depth <= 31 that is both default configurations. The library's choice stages exactly when the tree fits whole."""
    from tracer_b200 import Scene
    names = Scene.kernel_configs()
    info = scene.info
    auto = 0
    for c, cfg in enumerate(names):
        usable, staged = expected_staging(cfg, info["maxDepth"], info["topNodes"])
        if c < 2:
            assert usable, (name, cfg)
        if usable:
            assert scene.set_kernel_config(c) == staged, (name, cfg)
            if auto == 0 and c > 0 and staged > 0 and info["nInterior"] <= staged:
                auto = c
        else:
            with pytest.raises(Exception):
                scene.set_kernel_config(c)
    scene.set_kernel_config(-1)
    assert scene.kernel_config() == names[auto], (name, info)
    return [c for c, cfg in enumerate(names) if expected_staging(cfg, info["maxDepth"], info["topNodes"])[0]]


def _trace_everything(port, prim, scene, rays, rays_any, where, cfgs):
    """Closest-hit and any-hit against the oracle: reference-layout kernel, packed kernel in every configuration, hit16
    against pack_hit16, trq_expand_hits against the oracle's records. -> every packed-kernel result (for comparing two
    scenes byte for byte), and the deepest level the oracle's closest-hit traversal reached."""
    from tracer_b200 import rays_to_torch
    from .test_gpu_fuzz import _assert_records
    from .test_gpu_parity import assert_hits_equal, gpu_trace
    out = []
    level = 0
    for any_hit, r in ((False, rays), (True, rays_any)):
        want = port.trace(prim, r, any=any_hit, records=True, counters=True, nthreads=8)
        assert_hits_equal(gpu_trace(scene, r, any_hit, reflayout=True), want["hits"], f"{where} any={any_hit} reflayout", want["records"])
        d = rays_to_torch(r, f"cuda:{scene.device}")
        for c in cfgs:
            scene.set_kernel_config(c)
            at = f"{where} any={any_hit} cfg={c}"
            h = scene.hit(d, any=any_hit)
            got = h.cpu().numpy().view(L.hit_dtype).reshape(-1)
            assert_hits_equal(got, want["hits"], at, want["records"])
            h16 = scene.hit(d, any=any_hit, hit16=True).cpu().numpy().view(L.hit16_dtype).reshape(-1)
            assert np.array_equal(h16.view(np.uint8), L.pack_hit16(got).view(np.uint8)), at + " hit16"
            if not any_hit and c == cfgs[0]:
                _assert_records(scene, r, h, want, at)
            out.append(got)
        scene.set_kernel_config(-1)
        if not any_hit:
            level = int(want["counters"]["max_level"].max())
    return out, level


@pytest.mark.gpu
@pytest.mark.parametrize("name", TREES)
def test_caller_built_tree_matches_the_oracle(built, port, name):
    torch = _torch()
    from tracer_b200 import DevicePrimitive, Scene
    prim, topo, lv = tree_case(name)
    rng = np.random.default_rng(len(name))
    rays = tree_rays(rng, prim, lv)
    if name.startswith("comb"):
        rays = np.concatenate([rays, comb_rays(rng, lv)])
    rays_any = with_finite_tmax(rng, rays, lv)
    want_info = expected_info(prim)
    results = []
    for how in ("host", "device"):
        scene = Scene(prim if how == "host" else DevicePrimitive.from_host(prim, "cuda:0"), 0)
        for k, v in want_info.items():
            assert scene.info[k] == v, (name, how, k, scene.info[k], v)
        cfgs = _check_configurations(scene, f"{name} {how}")
        if name.startswith("spine"):                           # configuration 1 stages a prefix of the top block
            assert 0 < scene.set_kernel_config(1) < scene.info["nInterior"]
            scene.set_kernel_config(-1)
        results.append((scene.info,) + _trace_everything(port, prim, scene, rays, rays_any, f"{name} {how}", cfgs))
        if how == "host" and name.startswith("spine"):         # host-pointer path: the same bytes as the device path
            for any_hit, r in ((False, rays), (True, rays_any)):
                dev = scene.hit(torch.from_numpy(r.view(np.float32).reshape(-1, 8)).cuda(), any=any_hit).cpu().numpy()
                assert np.array_equal(scene.hit(r, any=any_hit).view(np.uint8), dev.view(np.uint8).reshape(-1))
                assert np.array_equal(scene.hit(r, any=any_hit, hit16=True).view(np.uint8),
                                      L.pack_hit16(dev.view(L.hit_dtype).reshape(-1)).view(np.uint8))
        scene.close()
    (host_info, host_out, level), (dev_info, dev_out, _) = results
    for k in ("nNode", "nInterior", "nLeaf", "maxDepth", "topNodes", "bytesPacked", "nTri", "nSphere", "nSquare", "nCube"):
        assert host_info[k] == dev_info[k], (name, k)
    assert len(host_out) == len(dev_out)
    for a, b in zip(host_out, dev_out):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), f"{name}: host-created and device-created scenes differ"
    if name.startswith(("comb", "spine")):                     # the deepest level is really reached
        assert want_info["maxDepth"] == MAX_DEPTH and level == MAX_DEPTH, name


@pytest.mark.gpu
@pytest.mark.parametrize("interior_left", [True, False])
def test_device_create_depth_boundary(built, interior_left):
    _torch()
    from tracer_b200 import DevicePrimitive, Scene
    from tracer_b200._lib import TrqError
    deep, _, _ = comb_prim(MAX_DEPTH, interior_left, how="random", seed=3)
    s = Scene(DevicePrimitive.from_host(deep, "cuda:0"), 0)
    assert s.info["maxDepth"] == MAX_DEPTH
    s.close()
    too_deep, _, _ = comb_prim(MAX_DEPTH + 1, interior_left, how="random", seed=3)
    with pytest.raises(TrqError) as e:
        Scene(DevicePrimitive.from_host(too_deep, "cuda:0"), 0)
    assert e.value.status == ERR_DEPTH


# --------------------------------------------------------------------------------------------------------- GPU: refit
def _one_two_leaves(n):
    lv = Leaves()
    lv.triangle([[0, 0, 0], [1, 0, 0], [0, 1, 0]])
    lv.triangle([[0, 0, 0], [1, 0, 0], [0, 0, 1]])
    t = Topo()
    if n == 1:
        t.root = t.add(leaf=0)
        lv.items = lv.items[:1]
    else:
        t.root = t.add(t.add(leaf=0), t.add(leaf=1))
    lo, hi = boxes(t, lv, "tight", None)
    prim = make_prim(t, lv, np.arange(len(t.leaf))[::-1].copy() if n == 2 else np.zeros(1, dtype=np.int64), lo, hi)
    if n == 1:
        prim = Primitive(triList=prim.triList[:3], idxList=prim.idxList[:3], bvhList=prim.bvhList)
    return prim


def _with_orphans(prim, rng):
    """Appends nodes the root does not reach, with every field in range: orphan triangle leaves (valid pIndex) whose parent
    field names a reachable interior node with two interior children -- several per level -- and one orphan interior
    node. A refit that climbed from the orphans would give those nodes a third arrival and merge them before one child
    subtree is done."""
    b = prim.bvhList
    e = np.full(b.size, -1)
    e[0] = 0
    stack = [0]
    while stack:
        i = stack.pop()
        if b["pType"][i] == L.BVH:
            for ch in (int(b["left"][i]), int(b["right"][i])):
                e[ch] = e[i] + 1
                stack.append(ch)
    inner = b["pType"] == L.BVH
    both = [i for i in np.nonzero(inner)[0] if inner[b["left"][i]] and inner[b["right"][i]]]
    targets = []
    for d in np.unique(e[both]):
        at = [i for i in both if e[i] == d]
        targets += list(rng.choice(at, min(4, len(at)), replace=False))
    assert len(targets) >= 20
    orphans = np.zeros(len(targets) + 1, dtype=L.bvh_dtype)
    orphans["pType"][:-1] = L.TRIANGLE
    orphans["pIndex"][:-1] = rng.integers(0, prim.nTri, len(targets))
    orphans["parent"][:-1] = targets
    orphans["mini"], orphans["maxi"] = b["mini"][0], b["maxi"][0]
    orphans["pType"][-1] = L.BVH                                  # an orphan interior node over two of the orphan leaves
    orphans["left"][-1], orphans["right"][-1] = b.size, b.size + 1
    orphans["parent"][-1] = targets[0]
    return Primitive(triList=prim.triList, idxList=prim.idxList, bvhList=np.concatenate([b, orphans]))


def refit_case(name):
    """-> (Primitive, moved vertices)."""
    rng = np.random.default_rng(sum(map(ord, name)))
    if name == "mixed_random":
        prim, _, _ = tree_case("split-random-inflated-mixed")
        verts = prim.triList.copy()
        verts["v"] += rng.uniform(-0.3, 0.3, verts["v"].shape).astype(f32)
    elif name == "comb31":
        prim, _, _ = comb_prim(MAX_DEPTH, interior_left=False, how="random", seed=5)
        verts = prim.triList.copy()
        verts["v"][:, 1:] += rng.uniform(-0.2, 0.2, verts["v"][:, 1:].shape).astype(f32)
        verts["v"][:, 0] -= f32(10)
    elif name in ("one_leaf", "two_leaves"):
        prim = _one_two_leaves(1 if name == "one_leaf" else 2)
        verts = prim.triList.copy()
        verts["v"] += np.array([3, -2, 5], dtype=f32)
        verts["v"][0] += f32(0.5)
    else:
        assert name == "unreachable"
        prim = _with_orphans(H.scene_soup(3000, seed=11, extent=0.05), rng)
        verts = prim.triList.copy()
        verts["v"] += np.array([1000, 700, 400], dtype=f32)
    return prim, verts


def _leaf_items(prim):
    """Leaves.items-like view of the geometry of a Primitive: (pType, pIndex, lo, hi) of every primitive."""
    lv = Leaves()
    if prim.nTri:
        p = prim.triList["v"][prim.idxList.reshape(-1, 3)]
        for k in range(prim.nTri):
            lv.items.append((L.TRIANGLE, k, p[k].min(0), p[k].max(0)))
    for t, arr in ((L.SPHERE, prim.sphereList), (L.SQUARE, prim.squareList)):
        for k in range(arr.size):
            lv.items.append((t, k, arr["box_mini"][k], arr["box_maxi"][k]))
    return lv


def _refit_rays(rng, prim):
    lv = _leaf_items(prim)
    return tree_rays(rng, prim, lv, n=2000), lv


def _info(scene):
    from tracer_b200._lib import SceneInfo, check
    i = SceneInfo()
    check(lib.trq_scene_info(scene._h, C.byref(i)), "trq_scene_info")
    return {k: getattr(i, k) for k, _ in SceneInfo._fields_}


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mixed_random", "comb31", "one_leaf", "two_leaves", "unreachable"])
def test_refit_of_caller_built_trees(built, port, name):
    """trq_scene_update_vertices against the oracle run on the tree refit with numpy (tests/util.refit_on_host), from a
    host and from a device vertex source; then the original vertices back."""
    torch = _torch()
    from tracer_b200 import Scene
    from .test_gpu_parity import assert_like_oracle, gpu_trace
    prim, verts = refit_case(name)
    moved = refit_on_host(prim, verts)
    rng = np.random.default_rng(7)
    rays, lv = _refit_rays(rng, moved)
    if name == "comb31":
        rays = np.concatenate([rays, comb_rays(rng, lv)])
    rays_any = with_finite_tmax(rng, rays, lv)
    old_rays = _refit_rays(rng, prim)[0]
    back = refit_on_host(prim, prim.triList)                   # inflated boxes come back as unions of their children
    scene = Scene(prim, 0)
    info = _info(scene)
    cfgs = [c for c, cfg in enumerate(Scene.kernel_configs()) if expected_staging(cfg, info["maxDepth"], info["topNodes"])[0]]
    for how in ("host", "device"):
        scene.update_vertices(verts if how == "host" else torch.from_numpy(verts.view(np.uint8).reshape(-1).copy()).cuda())
        assert _info(scene) == info
        _, level = _trace_everything(port, moved, scene, rays, rays_any, f"refit {name} ({how} vertices)", cfgs)
        if name == "comb31":
            assert level == MAX_DEPTH
        scene.update_vertices(prim.triList)                    # and back: the original geometry's answers return
        for any_hit in (False, True):
            assert_like_oracle(gpu_trace(scene, old_rays, any_hit), port, back, old_rays, any_hit, f"refit {name} back ({how})")
    scene.close()
