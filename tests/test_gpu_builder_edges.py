"""The GPU builder (trq_bvh_build_tree_gpu, trq_bvh_build_tree_device) against the host builder on leaves the scene
generators never make: signed zeros, infinite sides (NaN and +inf centroids), coordinates near +-FLT_MAX, denormals,
points, centroids on one line or one plane, lattice centroids on bucket edges, combs deeper than 64 levels and leaf
counts around the prefix scan's tiles.

Every leaf set is generated from a seed. The three builds must agree on status, nNode and maxDepth and give the same
node array (boxes compared by value); a tree that can be traced is traced, closest-hit and any-hit, against port.trace
on the host-built tree. The CPU tests at the end check that every generator still produces its edge case, so a GPU pass
cannot come from a generator that quietly stopped making it."""
import ctypes as C

import numpy as np
import pytest

from tracer_b200 import harness as H, layout as L
from tracer_b200._lib import ERR_DEPTH, check, lib

from .test_builder import check_tree
from .test_gpu_builder import assert_same_tree
from .test_gpu_parity import _torch, assert_hits_equal, gpu_trace

F = np.float32
NEG0 = F(-0.0)
AXES = "xyz"


# ---------------------------------------------------------------------------------------------------------------
# leaf sets: (triList, idxList, leaves, ray box). Leaves are triangle leaves over a soup, so every tree can be traced;
# where a set edits the boxes, the triangle inside may stick out of its box, which both tracers see alike.

def _soup(n, seed, extent=0.05):
    tri = np.zeros(3 * n, dtype=L.vertex_dtype)
    idx = np.zeros(3 * n, dtype=np.uint32)
    lib.trqh_make_soup(n, seed, extent, tri.ctypes.data, idx.ctypes.data)
    return tri, idx


def _leaves(tri, idx):
    n = idx.size // 3
    lv = np.zeros(n, dtype=L.bvh_dtype)
    check(lib.trq_bvh_build_nodes_triangles(tri.ctypes.data, idx.ctypes.data, n, 0, lv.ctypes.data), "leaves")
    return lv


UNIT = ((-0.2, -0.2, -0.2), (1.2, 1.2, 1.2))


def negzero_flat(axis, n=2000):
    """Every triangle flat in the plane axis = 0, every leaf with mini = maxi = -0.0 on that axis (as a caller's own
    boxes may have; trq_bvh_build_node's identity transform would make them +0.0)."""
    tri, idx = _soup(n, 40 + axis)
    tri["v"][:, axis] = NEG0
    lv = _leaves(tri, idx)
    lv["mini"][:, axis] = lv["maxi"][:, axis] = NEG0
    return tri, idx, lv, UNIT


def negzero_maxi(axis, seed, n=2000):
    """Geometry moved below 0 on `axis`; half of the leaves, in shuffled order, grow their maxi to -0.0."""
    tri, idx = _soup(n, seed)
    tri["v"][:, axis] -= F(1.1)
    lv = _leaves(tri, idx)
    lv["maxi"][np.random.default_rng(seed).permutation(n)[: n // 2], axis] = NEG0
    lo, hi = np.array(UNIT, dtype=np.float64)
    lo[axis], hi[axis] = -1.3, 0.1
    return tri, idx, lv, (tuple(lo), tuple(hi))


def negzero_mini(axis, seed, n=2000):
    """Geometry moved above 0 on `axis`; half of the leaves grow their mini to -0.0, the rest to a negative value."""
    rng = np.random.default_rng(seed)
    tri, idx = _soup(n, seed)
    tri["v"][:, axis] += F(0.1)
    lv = _leaves(tri, idx)
    perm = rng.permutation(n)
    lv["mini"][perm[: n // 2], axis] = NEG0
    lv["mini"][perm[n // 2:], axis] = -(rng.random(n - n // 2, dtype=F) * F(0.5) + F(0.01))
    return tri, idx, lv, UNIT


def infinite_sides(seed, n=3000, plus_inf=False, lead_warp=False):
    """10-30 % of the leaves, spread through the list, get mini = -inf (NaN centroid) or both sides infinite (NaN
    centroid) on one random axis; with plus_inf, maxi = +inf alone (+inf centroid) is a third choice. lead_warp: the
    first 32 leaves all have mini.x = -inf, so a whole warp of NaN x-centroids meets the reductions."""
    rng = np.random.default_rng(seed)
    tri, idx = _soup(n, seed)
    lv = _leaves(tri, idx)
    pick = rng.permutation(n)[: int((0.1 + 0.2 * rng.random()) * n)]
    axis = rng.integers(0, 3, pick.size)
    how = rng.integers(0, 3 if plus_inf else 2, pick.size)            # 0: mini = -inf, 1: both, 2: maxi = +inf
    lv["mini"][pick[how <= 1], axis[how <= 1]] = -np.inf
    lv["maxi"][pick[how >= 1], axis[how >= 1]] = np.inf
    if lead_warp:
        lv["mini"][:32, 0] = -np.inf
    return tri, idx, lv, UNIT


def one_inf_side_per_axis(seed, n=2000):
    """Three leaves, one per axis, with maxi = +inf on that axis: +inf centroids, but no two on the same axis. Every
    node holding one of them spans an infinite extent and takes the sort + median fallback with distinct keys."""
    rng = np.random.default_rng(seed)
    tri, idx = _soup(n, seed)
    lv = _leaves(tri, idx)
    lv["maxi"][rng.choice(n, 3, replace=False), [0, 1, 2]] = np.inf
    return tri, idx, lv, UNIT


def _boxes(rng, n, c, h):
    tri, idx = _soup(n, int(rng.integers(1 << 30)))
    lv = _leaves(tri, idx)
    lv["mini"], lv["maxi"] = (c - h).astype(F), (c + h).astype(F)
    return tri, idx, lv


def huge(seed, n=2000):
    """Centroids within +-1.6e38 and half-sides up to 1.6e38: box diagonals and areas overflow to inf, the centroid box
    stays finite."""
    rng = np.random.default_rng(seed)
    return _boxes(rng, n, rng.uniform(-1.6e38, 1.6e38, (n, 3)), rng.uniform(0, 1.6e38, (n, 3))) + (UNIT,)


def overflowing_centroids(seed, n=2000):
    """Centroids near -FLT_MAX and +FLT_MAX: the centroid box's extent itself overflows. On every axis the centroids
    are at least 1.6e35 apart, far above float32's spacing there, so the fallback's sort keys are distinct."""
    rng = np.random.default_rng(seed)
    step = 6.6e38 / n
    c = np.stack([rng.permutation(n) for _ in range(3)], 1) * step - 3.3e38 + rng.uniform(0, step / 2, (n, 3))
    return _boxes(rng, n, c, rng.uniform(0, step / 8, (n, 3))) + (UNIT,)


def denormal(seed, n=2000):
    """Every coordinate a denormal multiple of 2^-149, extents down to one denormal step (and some zero)."""
    rng = np.random.default_rng(seed)
    q = 2.0 ** -149
    lo = rng.integers(0, 1 << 20, (n, 3))
    tri, idx = _soup(n, seed)
    lv = _leaves(tri, idx)
    lv["mini"], lv["maxi"] = (lo * q).astype(F), ((lo + rng.integers(0, 1 << 12, (n, 3))) * q).astype(F)
    return tri, idx, lv, UNIT


def points(seed, n=2000):
    """Zero-extent boxes."""
    rng = np.random.default_rng(seed)
    p = rng.random((n, 3), dtype=F)
    return _boxes(rng, n, p, np.zeros_like(p)) + (UNIT,)


def _dyadic_boxes(rng, n, c):
    # c and the half-sides are multiples of 2^-13 below 1: mini + (maxi - mini) / 2 gives c back exactly
    return _boxes(rng, n, c, rng.integers(0, 64, (n, 3)) / 8192.0)


def line(seed, n=2000):
    """Every centroid on the diagonal x = y = z: the three extents tie in maximumExtent at every node."""
    rng = np.random.default_rng(seed)
    t = rng.choice(8192, n, replace=False) / 8192.0
    return _dyadic_boxes(rng, n, np.stack([t, t, t], 1)) + (UNIT,)


def plane(seed, n=2000):
    """Every centroid on the plane x = y: the x and y extents tie at every node."""
    rng = np.random.default_rng(seed)
    t = rng.choice(8192, n, replace=False) / 8192.0
    return _dyadic_boxes(rng, n, np.stack([t, t, rng.integers(0, 4096, n) / 8192.0], 1)) + (UNIT,)


def lattice_pairs(seed, n_distinct=900, n_pairs=300):
    """Integer centroids in [0, 10]^3, so 10 * relative() lands on bucket edges; n_pairs of them are shared by exactly
    two leaves (three or more are the documented exception)."""
    rng = np.random.default_rng(seed)
    cell = rng.choice(11 ** 3, n_distinct, replace=False)
    cell = np.concatenate([cell, cell[rng.choice(n_distinct, n_pairs, replace=False)]])
    c = np.stack([cell % 11, cell // 11 % 11, cell // 121], 1)[rng.permutation(cell.size)].astype(np.float64)
    tri, idx, lv = _boxes(rng, cell.size, c, rng.integers(0, 3, c.shape) * 0.25)
    tri["v"] *= F(10)                                                     # spread the soup over the lattice
    return tri, idx, lv, ((-1, -1, -1), (11, 11, 11))


# x-centroids base^k (k = lo..hi) as points on x, y and z in [0, 1]: interior depth of the host's tree
COMBS = {35: (11, 0, 36), 59: (11, -30, 30), 67: (16, -37, 31), 71: (11, -36, 36), 78: (11, -43, 36)}


def comb(depth, seed=1):
    base, lo, hi = COMBS[depth]
    x = np.array([float(base) ** k for k in range(lo, hi + 1)]).astype(F)
    n = x.size
    tri, idx = _soup(n, seed)
    lv = _leaves(tri, idx)
    lv["mini"][:, 0] = lv["maxi"][:, 0] = x[np.random.default_rng(seed).permutation(n)]
    lv["mini"][:, 1:], lv["maxi"][:, 1:] = 0, 1
    return tri, idx, lv, UNIT


def soup(n, seed=3):
    tri, idx = _soup(n, seed, 0.05 if n < 100_000 else 0.004)
    return tri, idx, _leaves(tri, idx), UNIT


EXACT = {f"negzero-flat-{AXES[a]}": (lambda a=a: negzero_flat(a)) for a in range(3)}
EXACT.update({f"negzero-maxi-{AXES[a]}-s{s}": (lambda a=a, s=s: negzero_maxi(a, s)) for a in range(3) for s in (1, 2)})
EXACT.update({f"negzero-mini-{AXES[a]}-s{s}": (lambda a=a, s=s: negzero_mini(a, s)) for a in range(3) for s in (1, 2)})
# NaN centroids always fall into bucket 0, and overflowing or underflowing areas make every SAH cost NaN (split 0):
# these trees grow deep, so each kind comes at a size that traces (depth <= 31) and at one past interior depth 31
EXACT.update({f"nan-centroids-s{s}": (lambda s=s: infinite_sides(s, 1000)) for s in (1, 2, 3, 4)})
EXACT["nan-centroids-leading-warp"] = lambda: infinite_sides(5, 1000, lead_warp=True)
EXACT["nan-centroids-deep"] = lambda: infinite_sides(6, 3000)
EXACT.update({"huge": lambda: huge(1, 200), "huge-deep": lambda: huge(2), "denormal": lambda: denormal(1, 200),
              "denormal-deep": lambda: denormal(2), "points": lambda: points(1),
              "line": lambda: line(1), "plane": lambda: plane(1), "lattice-pairs-s1": lambda: lattice_pairs(1),
              "lattice-pairs-s2": lambda: lattice_pairs(2)})
# nodes spanning an infinite centroid extent take the sort + median fallback; with distinct keys its result is unique
EXACT.update({f"inf-side-per-axis-s{s}": (lambda s=s: one_inf_side_per_axis(s)) for s in (1, 2)})
EXACT["overflowing-centroids"] = lambda: overflowing_centroids(2, 400)
EXACT["overflowing-centroids-deep"] = lambda: overflowing_centroids(1)
EXACT.update({f"comb-depth-{d}": (lambda d=d: comb(d)) for d in COMBS})
EXACT.update({f"soup-{n}": (lambda n=n: soup(n)) for n in (4095, 4096, 4097, 8191)})
LARGE = {f"soup-{n}": (lambda n=n: soup(n)) for n in (4_194_304, 5_000_000)}       # > 1024 scan tiles
# Many +inf centroids on one axis, beside NaN ones: the fallback sorts equal (+inf) and NaN keys, whose order std::sort
# leaves unspecified (include/tracer_rq.h). The trees may differ; both must be valid and give the same closest hits.
FALLBACK = {f"tied-inf-centroids-s{s}": (lambda s=s: infinite_sides(s, plus_inf=True)) for s in (1, 2)}


# ---------------------------------------------------------------------------------------------------------------
def centroids(lv):
    with np.errstate(invalid="ignore", over="ignore"):
        return lv["mini"] + (lv["maxi"] - lv["mini"]) / F(2)


def max_shared_centroid(lv):
    return int(np.unique(np.ascontiguousarray(centroids(lv)).view("V12").ravel(), return_counts=True)[1].max())


def build_three(leaves):
    """(status, nNode, maxDepth, nodes) of the host build, trq_bvh_build_tree_gpu and trq_bvh_build_tree_device."""
    torch = _torch()
    n = leaves.size
    out = []
    for gpu in (False, True):
        nodes = np.zeros(2 * n - 1, dtype=L.bvh_dtype)
        nodes[:n] = leaves
        nn, d = C.c_uint32(0xdead), C.c_uint32(0xdead)
        if gpu:
            rc = lib.trq_bvh_build_tree_gpu(nodes.ctypes.data, n, 0, C.byref(nn), C.byref(d))
        else:
            rc = lib.trq_bvh_build_tree(nodes.ctypes.data, n, C.byref(nn), C.byref(d))
        out.append((rc, nn.value, d.value, nodes))
    dev = torch.zeros((2 * n - 1) * L.bvh_dtype.itemsize, dtype=torch.uint8, device="cuda:0")
    dev[: n * L.bvh_dtype.itemsize] = torch.from_numpy(leaves.view(np.uint8).reshape(-1)).to(dev.device)
    nn, d = C.c_uint32(0xdead), C.c_uint32(0xdead)
    rc = lib.trq_bvh_build_tree_device(dev.data_ptr(), n, 0, C.byref(nn), C.byref(d))
    torch.cuda.synchronize()
    out.append((rc, nn.value, d.value, dev.cpu().numpy().view(L.bvh_dtype)))
    return out


def trace_both(port, tri, idx, tree, want_tree, box, seed, where, t_only=False):
    """Trace seeded random rays through a scene made of `tree` and compare with port.trace on `want_tree`."""
    from tracer_b200 import Scene
    from tracer_b200.scene import Primitive
    scene = Scene(Primitive(triList=tri, idxList=idx, bvhList=tree), 0)
    rays = H.random_rays(4000, seed=seed, lo=box[0], hi=box[1])
    for any_hit in (False, True):
        got = gpu_trace(scene, rays, any_hit)
        want = port.trace(Primitive(triList=tri, idxList=idx, bvhList=want_tree), rays, any=any_hit, records=True, nthreads=8)
        want, recs = want["hits"], want["records"]
        if t_only:
            assert np.array_equal(got["flags"] & 1, want["flags"] & 1), f"{where} any={any_hit}: hit flags differ"
            if not any_hit:
                assert np.array_equal(got["t"].view(np.uint32), want["t"].view(np.uint32)), f"{where}: closest t differs"
        else:
            assert_hits_equal(got, want, f"{where} any={any_hit}", recs)
    scene.close()


def _exact(port, name, make, byte_exact=False):
    tri, idx, lv, box = make()
    n = lv.size
    (hrc, hn, hd, h), (grc, gn, gd, g), (drc, dn, dd, dv) = build_three(lv)
    assert (grc, gn, gd) == (hrc, hn, hd), f"{name}: gpu (status, nNode, maxDepth) {(grc, gn, gd)} vs host {(hrc, hn, hd)}"
    assert (drc, dn, dd) == (hrc, hn, hd), f"{name}: device (status, nNode, maxDepth) {(drc, dn, dd)} vs host {(hrc, hn, hd)}"
    if byte_exact:
        assert np.array_equal(g.view(np.uint8), h.view(np.uint8)), f"{name}: gpu node array differs from the host's"
        assert np.array_equal(dv.view(np.uint8), h.view(np.uint8)), f"{name}: device node array differs from the host's"
    else:
        assert_same_tree(h, g)
        assert_same_tree(h, dv)
    if hrc == ERR_DEPTH:
        assert check_tree(g, n) == gd > 31, name
    else:
        assert hrc == 0, name
        trace_both(port, tri, idx, g, h, box, n + 7, name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(EXACT))
def test_gpu_builds_equal_host_build(built, port, name):
    _exact(port, name, EXACT[name])


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(LARGE))
def test_gpu_builds_equal_host_build_past_1024_scan_tiles(built, port, name):
    _exact(port, name, LARGE[name], byte_exact=True)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FALLBACK))
def test_gpu_fallback_nodes_build_valid_trees(built, port, name):
    tri, idx, lv, box = FALLBACK[name]()
    n = lv.size
    (hrc, hn, hd, h), (grc, gn, gd, g), (drc, dn, dd, dv) = build_three(lv)
    assert gn == hn and (drc, dn, dd) == (grc, gn, gd), f"{name}: host {(hrc, hn, hd)} gpu {(grc, gn, gd)} device {(drc, dn, dd)}"
    assert np.array_equal(dv.view(np.uint8), g.view(np.uint8)), f"{name}: the two GPU builds differ"
    assert check_tree(h, n) == hd and check_tree(g, n) == gd, name          # the depths may differ, not their meaning
    assert (hrc, grc) == (ERR_DEPTH if hd > 31 else 0, ERR_DEPTH if gd > 31 else 0), name
    if grc == 0:
        trace_both(port, tri, idx, g, g, box, n + 7, f"{name} (GPU tree)")
        if hrc == 0:                                                      # boxes still hold their triangles
            trace_both(port, tri, idx, g, h, box, n + 7, f"{name} (host tree)", t_only=True)


# ---------------------------------------------------------------------------------------------------------------
# CPU: the generators make what they claim, on the host builder

def _host(lv):
    n = lv.size
    nodes = np.zeros(2 * n - 1, dtype=L.bvh_dtype)
    nodes[:n] = lv
    nn, d = C.c_uint32(0), C.c_uint32(0)
    rc = lib.trq_bvh_build_tree(nodes.ctypes.data, n, C.byref(nn), C.byref(d))
    return rc, nn.value, d.value, nodes


def _is_neg0(a):
    return np.asarray(a, dtype=F).view(np.uint32) == 0x80000000


@pytest.mark.parametrize("depth", list(COMBS))
def test_combs_have_their_depth_on_the_host(built, depth):
    _, _, lv, _ = comb(depth)
    assert np.unique(lv["mini"][:, 0]).size == lv.size
    rc, nn, d, nodes = _host(lv)
    assert rc == ERR_DEPTH and nn == 2 * lv.size - 1 and d == depth
    assert check_tree(nodes, lv.size) == depth                            # the complete tree comes back with the error
    if depth == 78:
        assert (lv["mini"][:, 0] < np.finfo(F).tiny).sum() > 0            # float32 denormal centroids


def test_edge_generators_make_their_edge(built):
    for a in range(3):
        lv = negzero_flat(a)[2]
        assert _is_neg0(lv["mini"][:, a]).all() and _is_neg0(lv["maxi"][:, a]).all()
        for s in (1, 2):
            lv = negzero_maxi(a, s)[2]
            m = lv["maxi"][:, a]
            assert _is_neg0(m).sum() == lv.size // 2 and (m[~_is_neg0(m)] < 0).all()
            m = negzero_mini(a, s)[2]["mini"][:, a]
            assert _is_neg0(m).sum() == lv.size // 2 and (m[~_is_neg0(m)] < 0).all()
    for s in (1, 2, 3, 4, 6):
        c = centroids(infinite_sides(s, 1000 if s < 6 else 3000)[2])
        share = np.isnan(c).any(1).mean()
        assert 0.1 <= share <= 0.3 and np.isfinite(c[~np.isnan(c)]).all()
    assert np.isnan(centroids(infinite_sides(5, 1000, lead_warp=True)[2])[:32, 0]).all()
    for s in (1, 2):
        c = centroids(infinite_sides(s, plus_inf=True)[2])
        assert (np.isposinf(c).sum(0) > 1).all() and np.isnan(c).any(), "tied +inf keys beside NaN keys"
        c = centroids(one_inf_side_per_axis(s)[2])
        assert (np.isposinf(c).sum(0) == 1).all() and np.isfinite(c[~np.isposinf(c)]).all()
    with np.errstate(over="ignore"):
        lv = huge(1)[2]
        c = centroids(lv)
        assert np.isfinite(c).all() and np.isfinite(c.max(0) - c.min(0)).all()
        assert np.isinf(lv["maxi"].max(0) - lv["mini"].min(0)).all()       # bucket diagonals overflow
        for args in ((1,), (2, 400)):
            c = centroids(overflowing_centroids(*args)[2])
            assert np.isfinite(c).all() and np.isinf(c.max(0) - c.min(0)).all()
            assert all(np.unique(c[:, k]).size == c.shape[0] for k in range(3)), "distinct sort keys"
    lv = denormal(1)[2]
    ext = lv["maxi"] - lv["mini"]
    assert (lv["maxi"] < np.finfo(F).tiny).all() and ((ext > 0) & (ext < np.finfo(F).tiny)).all(1).any()
    lv = points(1)[2]
    assert np.array_equal(lv["mini"], lv["maxi"])
    c = centroids(line(1)[2])
    assert (c[:, 0] == c[:, 1]).all() and (c[:, 1] == c[:, 2]).all()
    c = centroids(plane(1)[2])
    assert (c[:, 0] == c[:, 1]).all() and not (c[:, 1] == c[:, 2]).all()
    for s in (1, 2):
        lv = lattice_pairs(s)[2]
        c = centroids(lv)
        assert (c == np.round(c)).all() and c.min() == 0 and c.max() == 10 and max_shared_centroid(lv) == 2
    for name, make in EXACT.items():                                      # >= 3 leaves on one centroid: the exception
        if not name.startswith("comb"):
            assert max_shared_centroid(make()[2]) <= 2, name


@pytest.mark.parametrize("name", [k for k in EXACT if not k.startswith("comb")])
def test_edge_sets_build_on_the_host(built, name):
    _, _, lv, _ = EXACT[name]()
    rc, nn, d, nodes = _host(lv)
    assert nn == 2 * lv.size - 1 and check_tree(nodes, lv.size) == d
    assert (rc, d > 31) == ((ERR_DEPTH, True) if name.endswith("-deep") else (0, False))
