"""CPU: the Morton-order builder's host restatement (trq_bvh_build_tree_morton) pinned against the rules written again
with numpy (tests/morton_util.py), byte for byte: soups, mixed leaf kinds, the builder edge sets of
test_gpu_builder_edges (signed zeros, infinite sides, overflowing centroids, denormals, points, lines, planes, lattice
ties, combs), a forced code chain that only the depth clamp keeps at depth 31, and port.trace through its trees."""
import ctypes as C

import numpy as np
import pytest

from tracer_b200 import Primitive, harness as H, layout as L
from tracer_b200._lib import ERR_INVALID, lib

from .morton_util import (QMAX, chain_points, check_morton_structure, host_morton, mixed_leaves, morton_codes, morton_tree,
                          point_leaves, quantise_axis, reference_cornell_leaves)
from .test_gpu_builder_edges import COMBS, EXACT, comb, soup

F = np.float32


def _pinned(leaves, name):
    rc, nn, depth, got = host_morton(leaves)
    assert (rc, nn) == (0, 2 * leaves.size - 1), (name, rc, lib.trq_last_error_string())
    want, want_depth, order = morton_tree(leaves)
    bad = np.nonzero(got.view("V64") != want.view("V64"))[0]
    assert bad.size == 0, f"{name}: {bad.size} nodes differ from the numpy rules, first {bad[:4]}: {got[bad[:1]]} vs {want[bad[:1]]}"
    assert depth == want_depth <= 31, (name, depth, want_depth)
    assert check_morton_structure(got, leaves, order) == depth, name
    return got, depth


@pytest.mark.parametrize("n", [1, 2, 3, 5, 17, 100, 1000, 4097])
def test_soups_equal_the_numpy_rules(built, n):
    _pinned(soup(n, seed=n + 1)[2], f"soup-{n}")


@pytest.mark.parametrize("seed", [1, 2])
def test_mixed_leaf_kinds_equal_the_numpy_rules(built, seed):
    _, lv = mixed_leaves(seed)
    assert set(lv["pType"].tolist()) == {L.SPHERE, L.SQUARE, L.CUBE, L.TRIANGLE}
    _pinned(lv, f"mixed-s{seed}")
    _pinned(reference_cornell_leaves()[1], "reference-cornell")


@pytest.mark.parametrize("name", list(EXACT))
def test_builder_edge_sets_equal_the_numpy_rules(built, name):
    _pinned(EXACT[name]()[2], name)


@pytest.mark.parametrize("depth", list(COMBS))
def test_combs_the_sah_builder_refuses_build_within_depth_31(built, depth):
    lv = comb(depth)[2]
    _, d = _pinned(lv, f"comb-{depth}")
    assert d <= 31


@pytest.mark.parametrize("copies", [1, 64])
def test_depth_clamp_keeps_a_forced_chain_at_depth_31(built, copies):
    lv = point_leaves(chain_points(copies))
    n = lv.size
    assert n & (n - 1) == 0
    codes = morton_codes(lv)
    single = codes[(codes & (codes - np.uint64(1))) == 0]
    assert np.unique(single).size == 63 and (codes == np.uint64((1 << 63) - 1)).sum() == copies
    assert morton_tree(lv, clamp=False)[1] > 40, "without the clamp the chain is deeper than the trail"
    got, depth = _pinned(lv, f"chain x{copies}")
    assert depth == 31
    leaves = got[1:n + 1]
    assert np.array_equal(np.sort(leaves["pIndex"]), np.arange(n))


def test_quantisation_rule_on_special_values(built):
    inf, nan = np.inf, np.nan
    assert list(quantise_axis([nan, inf, -inf, 0.0, 1.0])) == [QMAX, QMAX, 0, 0, QMAX]
    assert list(quantise_axis([nan, inf, -inf])) == [QMAX, QMAX, 0]                   # no finite component
    assert list(quantise_axis([2.5, 2.5, nan])) == [0, 0, QMAX]                       # zero extent
    assert list(quantise_axis([-3e38, 3e38, 0.0])) == [0, 0, 0]                       # extent overflows
    assert list(quantise_axis([-0.0, 0.0, 2.0 ** -149, 2.0 ** -148])) == [0, 0, 1 << 20, QMAX]   # denormal extent
    # the same values through the host restatement: a code is visible in the tree as its leaf's sorted place
    vals = np.array([nan, inf, -inf, -0.0, 0.0, 1e-45, 3.4028235e38, -3.4028235e38, 1.0], dtype=F)
    pts = np.stack([vals, vals[::-1], np.roll(vals, 3)], 1)
    _pinned(point_leaves(pts), "special values")


def test_oracle_traces_morton_trees_like_sah_trees(built, port):
    """Same hit flags and t (closest and any hit); primitive ids may differ only where two primitives tie at t."""
    for n, seed in ((3000, 1), (1500, 2)):
        prim = H.scene_soup(n, seed=seed, extent=0.05)
        lv = prim.bvhList[1:n + 1].copy()
        rc, _, _, tree = host_morton(lv)
        assert rc == 0
        mprim = Primitive(triList=prim.triList, idxList=prim.idxList, bvhList=tree)
        rays = H.random_rays(4000, seed=seed + 10)
        for any_hit in (False, True):
            a = port.trace(prim, rays, any=any_hit, nthreads=8)["hits"]
            b = port.trace(mprim, rays, any=any_hit, nthreads=8)["hits"]
            assert np.array_equal(a["flags"] & 1, b["flags"] & 1), (n, any_hit)
            if not any_hit:
                assert np.array_equal(a["t"].view(np.uint32), b["t"].view(np.uint32)), n
                differ = (a["pIndex"] != b["pIndex"]) & ((a["flags"] & 1) != 0)
                assert differ.sum() <= 2, (n, differ.sum())


def test_host_restatement_refuses_bad_arguments(built):
    nn, d = C.c_uint32(0), C.c_uint32(7)
    lv = np.zeros(1, dtype=L.bvh_dtype)
    assert lib.trq_bvh_build_tree_morton(None, 4, C.byref(nn), C.byref(d)) == ERR_INVALID
    assert lib.trq_bvh_build_tree_morton(lv.ctypes.data, 0, C.byref(nn), C.byref(d)) == ERR_INVALID
    assert lib.trq_bvh_build_tree_morton(lv.ctypes.data, 0x40000000, C.byref(nn), C.byref(d)) == ERR_INVALID
    assert b"too many" in lib.trq_last_error_string()


def test_python_method_argument(built):
    from tracer_b200 import BVHBuilder
    prim = H.scene_soup(500, seed=4, extent=0.05)
    b = BVHBuilder()
    b.buildNodesTriangles(prim.triList, prim.idxList)
    tree = b.buildTree(method="morton")
    assert tree.tobytes() == host_morton(prim.bvhList[1:501].copy())[3].tobytes() and b.maxDepth <= 31
    assert b.buildTree().tobytes() == prim.bvhList.tobytes()                          # the default stays the SAH builder
    for bad in ("lbvh", "SAH", None):
        with pytest.raises(ValueError):
            b.buildTree(method=bad)
    with pytest.raises(ValueError):
        BVHBuilder().buildTree(method="morton")                                       # no leaves
