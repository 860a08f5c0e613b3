"""The Morton-order builder on the GPU (trq_bvh_build_tree_morton_device, trq_scene_rebuild with TRQ_BUILD_MORTON,
BVHBuilder / DevicePrimitive.build / Scene.rebuild with method="morton").

The device tree must equal the host restatement (trq_bvh_build_tree_morton, itself pinned against numpy in
test_morton_build_cpu.py) byte for byte; scenes made from Morton trees must trace like port.trace in every kernel
configuration; a Morton rebuild must equal its host restatement, leave the scene as a fresh device create of the new tree
would be, refit like any other tree, rebuild scenes the SAH builder cannot, and leave the scene intact when refused."""
import ctypes as C

import numpy as np
import pytest

from tracer_b200 import Primitive, harness as H, layout as L
from tracer_b200._lib import ERR_DEPTH, ERR_INVALID, TrqError, check, lib

from .morton_util import (chain_points, check_morton_structure, host_morton, mixed_leaves, morton_codes, morton_rebuild_on_host,
                          point_leaves, rebuild_leaves, reference_cornell_leaves)
from .test_gpu_builder_edges import COMBS, EXACT, LARGE, soup
from .test_gpu_parity import assert_hits_equal, assert_like_oracle, gpu_trace, oracle
from .test_gpu_tree_shapes import (_check_configurations, _leaf_items, _trace_everything, comb_rays, refit_case, tree_rays,
                                   with_finite_tmax)
from .update_util import update_on_host
from .util import refit_on_host

pytestmark = pytest.mark.gpu
f32 = np.float32


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def device_morton(leaves):
    """trq_bvh_build_tree_morton_device -> (status, nNode, maxDepth, nodes)."""
    torch = _torch()
    n = leaves.size
    d = torch.full(((2 * n - 1) * 64,), 0xA5, dtype=torch.uint8, device="cuda:0")
    d[: n * 64] = torch.from_numpy(leaves.view(np.uint8).reshape(-1).copy()).cuda()
    nn, depth = C.c_uint32(0xdead), C.c_uint32(0xdead)
    rc = lib.trq_bvh_build_tree_morton_device(d.data_ptr(), n, 0, C.byref(nn), C.byref(depth))
    torch.cuda.synchronize()
    return rc, nn.value, depth.value, d.cpu().numpy().view(L.bvh_dtype)


def _special_points():
    vals = np.array([np.nan, np.inf, -np.inf, -0.0, 0.0, 1e-45, 3.4028235e38, -3.4028235e38, 1.0], dtype=f32)
    return point_leaves(np.stack([vals, vals[::-1], np.roll(vals, 3)], 1))


def _c3_leaves():
    tri, idx = H.cornell_triangle_soup(with_teapot=True, mesh_levels=2, with_coatball=True)
    n = idx.size // 3
    lv = np.zeros(n, dtype=L.bvh_dtype)
    check(lib.trq_bvh_build_nodes_triangles(tri.ctypes.data, idx.ctypes.data, n, 0, lv.ctypes.data), "leaves")
    return lv


SETS = {f"soup-{n}": (lambda n=n: soup(n, seed=n)[2]) for n in (2, 3, 33, 1000, 50_000)}
SETS.update({f"mixed-s{s}": (lambda s=s: mixed_leaves(s)[1]) for s in (1, 2)})
SETS["reference-cornell"] = lambda: reference_cornell_leaves()[1]
SETS.update({name: (lambda make=make: make()[2]) for name, make in EXACT.items()})
SETS.update({f"chain-x{c}": (lambda c=c: point_leaves(chain_points(c))) for c in (1, 64)})
SETS["special-values"] = _special_points
SETS["c3"] = _c3_leaves
SETS.update({name: (lambda make=make: make()[2]) for name, make in LARGE.items()})     # > 1024 scan tiles


@pytest.mark.parametrize("name", list(SETS))
def test_device_build_equals_host_restatement(built, name):
    _torch()
    lv = SETS[name]()
    hrc, hn, hd, h = host_morton(lv)
    drc, dn, dd, d = device_morton(lv)
    assert (drc, dn, dd) == (hrc, hn, hd) == (0, 2 * lv.size - 1, hd), (name, (drc, dn, dd), (hrc, hn, hd), lib.trq_last_error_string())
    bad = np.nonzero(d.view("V64") != h.view("V64"))[0]
    assert bad.size == 0, f"{name}: {bad.size} nodes differ, first {bad[:4]}: device {d[bad[:1]]} host {h[bad[:1]]}"
    assert hd <= 31
    if lv.size <= 60_000:
        order = np.argsort(morton_codes(lv), kind="stable")
        assert check_morton_structure(d, lv, order) == dd, name


def test_single_leaf_and_refusals(built):
    torch = _torch()
    lv = soup(1, seed=3)[2]
    rc, nn, depth, d = device_morton(lv)
    assert (rc, nn, depth) == (0, 1, 0) and d["parent"][0] == 0 and d[0:1].tobytes() == host_morton(lv)[3].tobytes()
    buf = torch.zeros(64 * 3, dtype=torch.uint8, device="cuda:0")
    nn, dp = C.c_uint32(0), C.c_uint32(9)
    assert lib.trq_bvh_build_tree_morton_device(None, 2, 0, C.byref(nn), C.byref(dp)) == ERR_INVALID and dp.value == 0
    assert lib.trq_bvh_build_tree_morton_device(buf.data_ptr(), 0, 0, C.byref(nn), C.byref(dp)) == ERR_INVALID
    assert lib.trq_bvh_build_tree_morton_device(buf.data_ptr(), 0x40000000, 0, C.byref(nn), C.byref(dp)) == ERR_INVALID
    assert lib.trq_bvh_build_tree_morton_device(buf.data_ptr(), 2, 4096, C.byref(nn), C.byref(dp)) == ERR_INVALID
    assert b"out of range" in lib.trq_last_error_string()


def test_python_entry_points(built):
    torch = _torch()
    from tracer_b200 import BVHBuilder, DevicePrimitive
    prim = H.scene_reference_cornell()
    n = (prim.bvhList.size + 1) // 2
    want = host_morton(reference_cornell_leaves()[1])[3]
    dprim = DevicePrimitive.build(*(None if a.size == 0 else torch.from_numpy(a.view(np.uint8).reshape(-1).copy()).cuda()
                                    for a in (prim.sphereList, prim.squareList, prim.cubeList, prim.triList, prim.idxList)),
                                  method="morton")
    assert dprim.arrays["bvhList"].cpu().numpy().tobytes() == want.tobytes() and dprim.maxDepth <= 31
    b = BVHBuilder()
    b._chunks.append(prim.bvhList[1:n + 1].copy())
    assert b.buildTree(gpu=0, method="morton").tobytes() == want.tobytes()
    assert b.buildTreeDevice(0, method="morton").cpu().numpy().tobytes() == want.tobytes()
    for bad in ("lbvh", None):
        with pytest.raises(ValueError):
            b.buildTreeDevice(0, method=bad)
        with pytest.raises(ValueError):
            DevicePrimitive.build(triList=dprim.arrays["triList"], idxList=dprim.arrays["idxList"], method=bad)


# ------------------------------------------------------------------------------------------- scenes of Morton trees
def _morton_scene_cases():
    """-> name: () -> (Primitive over a Morton tree, "comb" when comb rays are wanted, else None)."""
    cases = {}
    cases["soup"] = lambda: (morton_rebuild_on_host(H.scene_soup(3000, seed=5, extent=0.05)), None)
    cases["reference-cornell"] = lambda: (morton_rebuild_on_host(H.scene_reference_cornell()), None)

    def mixed():
        lv, leaves = mixed_leaves(3, 300)
        arrays = lv.arrays()
        return Primitive(**arrays, bvhList=host_morton(leaves)[3]), None
    cases["mixed"] = mixed

    def comb35():
        from .test_gpu_builder_edges import comb
        tri, idx, leaves, _ = comb(35)
        p = Primitive(triList=tri, idxList=idx, bvhList=host_morton(leaves)[3])
        return p, "comb"
    cases["comb-35"] = comb35
    return cases


CASES = _morton_scene_cases()


@pytest.mark.parametrize("name", list(CASES))
def test_scenes_of_morton_trees_trace_like_the_oracle(built, port, name):
    _torch()
    from tracer_b200 import DevicePrimitive, Scene
    prim, extra = CASES[name]()
    rng = np.random.default_rng(len(name))
    lv = _leaf_items(prim)
    if prim.cubeList.size:                                  # cube leaves: their world boxes come from the tree's leaves
        for k in np.nonzero(prim.bvhList["pType"] == L.CUBE)[0]:
            lv.items.append((L.CUBE, int(prim.bvhList["pIndex"][k]), prim.bvhList["mini"][k], prim.bvhList["maxi"][k]))
    rays = tree_rays(rng, prim, lv, n=2000)
    if extra == "comb":
        rays = np.concatenate([rays, comb_rays(rng, lv)])
    rays_any = with_finite_tmax(rng, rays, lv)
    for how in ("host", "device"):
        scene = Scene(prim if how == "host" else DevicePrimitive.from_host(prim, "cuda:0"), 0)
        assert scene.bvh().tobytes() == prim.bvhList.tobytes() and scene.info["maxDepth"] <= 31
        cfgs = _check_configurations(scene, f"{name} {how}")
        _trace_everything(port, prim, scene, rays, rays_any, f"morton {name} {how}", cfgs)
        scene.close()


# ----------------------------------------------------------------------------------------------------- Morton rebuilds
def _moved(prim, how, rng):
    v = prim.triList.copy()
    if how == "jitter":
        v["v"] += rng.uniform(-0.002, 0.002, v["v"].shape).astype(f32)
    else:                                                   # every triangle takes another one's place
        tri = v.reshape(-1, 3)
        v = np.ascontiguousarray(tri[rng.permutation(tri.shape[0])].reshape(-1))
    return v


def _fresh_info(rebuilt):
    from tracer_b200 import DevicePrimitive, Scene
    s = Scene(DevicePrimitive.from_host(rebuilt, "cuda:0"), 0)
    info = dict(s.info)
    s.close()
    return info


@pytest.mark.parametrize("how", ["jitter", "permute"])
@pytest.mark.parametrize("source", ["host", "device"])
def test_morton_rebuild_after_motion(built, port, how, source):
    torch = _torch()
    from tracer_b200 import Scene
    rng = np.random.default_rng(len(how) * 7 + len(source))
    prim = H.scene_soup(20000, seed=6, extent=0.01)
    verts = _moved(prim, how, rng)
    want = morton_rebuild_on_host(prim, verts)
    scene = Scene(prim, 0)
    scene.rebuild(verts if source == "host" else torch.from_numpy(verts.view(np.uint8).reshape(-1).copy()).cuda(), method="morton")
    assert scene.bvh().tobytes() == want.bvhList.tobytes()
    assert scene.info == _fresh_info(want)
    cfgs = _check_configurations(scene, f"morton rebuild {how} {source}")
    rays = H.random_rays(6000, seed=11)
    rays_any = with_finite_tmax(rng, rays, _leaf_items(want))
    _trace_everything(port, want, scene, rays, rays_any, f"morton rebuild {how} ({source} vertices)", cfgs)
    again = verts.copy()                                    # a refit of the Morton tree follows the vertices
    again["v"] += rng.uniform(-0.003, 0.003, again["v"].shape).astype(f32)
    scene.update_vertices(again)
    refit = refit_on_host(want, again)
    assert scene.bvh().tobytes() == refit.bvhList.tobytes()
    for any_hit in (False, True):
        assert_like_oracle(gpu_trace(scene, rays, any_hit), port, refit, rays, any_hit, f"refit any={any_hit}")
    scene.rebuild(method="sah")                             # and the SAH builder takes it back
    from .rebuild_util import rebuild_on_host
    assert scene.bvh().tobytes() == rebuild_on_host(refit).bvhList.tobytes()
    scene.close()


def test_morton_rebuild_then_update_primitives(built, port):
    _torch()
    from tracer_b200 import Scene
    prim = H.scene_reference_cornell()
    rng = np.random.default_rng(4)
    verts = prim.triList.copy()
    verts["v"] += rng.uniform(-0.05, 0.05, verts["v"].shape).astype(f32)
    want = morton_rebuild_on_host(prim, verts)
    scene = Scene(prim, 0)
    scene.rebuild(verts, method="morton")
    assert scene.bvh().tobytes() == want.bvhList.tobytes() and scene.info == _fresh_info(want)
    spheres = prim.sphereList.copy()
    spheres["box_mini"] -= f32(0.1)
    cubes = prim.cubeList.copy()
    cubes["model"][:, 12] += f32(0.05)
    scene.update_primitives(spheres=spheres, cubes=cubes)
    moved = update_on_host(want, spheres=spheres, cubes=cubes)
    assert scene.bvh().tobytes() == moved.bvhList.tobytes()
    rays = H.cornell_camera_rays(160, 90)
    for any_hit in (False, True):
        got, (want, recs) = gpu_trace(scene, rays, any_hit), oracle(port, moved, rays, any_hit)
        assert_hits_equal(got, want, f"moved any={any_hit}", recs)
        miss = (want["flags"] & 1) == 0                          # and the u / v bytes of the misses
        for k in ("u", "v"):
            assert np.array_equal(got[k][miss].view(np.uint32), want[k][miss].view(np.uint32)), (k, any_hit)
    scene.close()


@pytest.mark.parametrize("name", ["unreachable", "one_leaf", "two_leaves", "comb31"])
def test_morton_rebuild_of_caller_built_trees(built, port, name):
    """Over the leaves the root reaches: a tree with unreachable nodes shrinks to 2n - 1 nodes."""
    _torch()
    from tracer_b200 import Scene
    prim, verts = refit_case(name)
    want = morton_rebuild_on_host(prim, verts)
    n_leaf = rebuild_leaves(prim).size
    scene = Scene(prim, 0)
    scene.rebuild(verts, method="morton")
    got = scene.bvh()
    assert got.tobytes() == want.bvhList.tobytes(), name
    assert scene.info["nNode"] == got.size == 2 * n_leaf - 1, name
    if name == "unreachable":
        assert prim.bvhList.size > got.size
    assert scene.info == _fresh_info(want), name
    cfgs = _check_configurations(scene, name) if scene.info["nInterior"] else [0]
    rng = np.random.default_rng(sum(map(ord, name)))
    lv = _leaf_items(want)
    rays = tree_rays(rng, want, lv, n=2000)
    _trace_everything(port, want, scene, rays, with_finite_tmax(rng, rays, lv), f"morton rebuild {name}", cfgs)
    scene.close()


def test_comb_the_sah_rebuild_refuses_rebuilds_with_morton(built, port):
    _torch()
    from tracer_b200 import Scene
    base, lo, hi = COMBS[35]
    x = np.array([float(base) ** k for k in range(lo, hi + 1)]).astype(f32)
    prim = H.scene_soup(x.size, seed=2, extent=0.05)
    comb = prim.triList.copy()                              # triangle i flat at x = 11^perm(i), spanning [0, 1] in y and z
    comb["v"] = np.tile(np.array([[0, 0, 0], [0, 1, 0], [0, 0, 1]], dtype=f32), (x.size, 1))
    comb["v"][:, 0] = np.repeat(x[np.random.default_rng(1).permutation(x.size)], 3)
    scene = Scene(prim, 0)
    rays = H.random_rays(5000, seed=3)
    bvh, info = scene.bvh().tobytes(), dict(scene.info)
    with pytest.raises(TrqError) as e:
        scene.rebuild(comb)
    assert e.value.status == ERR_DEPTH
    assert scene.bvh().tobytes() == bvh and scene.info == info
    scene.rebuild(comb, method="morton")
    want = morton_rebuild_on_host(prim, comb)
    assert scene.bvh().tobytes() == want.bvhList.tobytes() and scene.info == _fresh_info(want) and scene.info["maxDepth"] <= 31
    lv = _leaf_items(want)
    rng = np.random.default_rng(5)
    rays = np.concatenate([rays, comb_rays(rng, lv), tree_rays(rng, want, lv, n=1000)])
    cfgs = _check_configurations(scene, "comb-35 morton rebuild")
    _trace_everything(port, want, scene, rays, with_finite_tmax(rng, rays, lv), "comb-35 morton rebuild", cfgs)
    scene.close()


def test_refused_morton_rebuild_leaves_the_scene_intact(built):
    _torch()
    from tracer_b200 import Scene
    prim = H.scene_soup(2000, seed=9, extent=0.05)
    scene = Scene(prim, 0)
    rays = H.random_rays(3000, seed=1)
    bvh, info, before = scene.bvh().tobytes(), dict(scene.info), gpu_trace(scene, rays)
    for bad in ("lbvh", "Morton", None, 1):
        with pytest.raises(ValueError):
            scene.rebuild(method=bad)
        with pytest.raises(ValueError):
            scene.rebuild(prim.triList, method=bad)
    v = prim.triList
    assert lib.trq_scene_rebuild(scene._h, v.ctypes.data, v.size - 1, L.HOST_PTRS | L.BUILD_MORTON) == ERR_INVALID
    assert lib.trq_scene_rebuild(None, None, 0, L.BUILD_MORTON) == ERR_INVALID
    assert scene.bvh().tobytes() == bvh and scene.info == info
    assert gpu_trace(scene, rays).tobytes() == before.tobytes()
    scene.close()


def test_morton_rebuild_waits_for_traces_in_flight(built):
    """A large trace queued on a side stream just before a Morton rebuild returns the answers of the tree before it."""
    torch = _torch()
    from tracer_b200 import Scene, rays_to_torch
    prim = H.scene_soup(300_000, seed=8, extent=0.004)
    scene = Scene(prim, 0)
    rays = rays_to_torch(H.random_rays(1 << 23, seed=4), "cuda:0")
    want = scene.hit(rays)
    torch.cuda.synchronize()
    moved = _moved(prim, "permute", np.random.default_rng(2))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        got = scene.hit(rays, stream=side.cuda_stream)
    scene.rebuild(moved, method="morton")
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    after = scene.hit(rays)
    torch.cuda.synchronize()
    assert not torch.equal(after, want)
    scene.close()
