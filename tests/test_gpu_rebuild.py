"""Device leaves and in-place scene rebuilds (trq_bvh_build_nodes_triangles_device, trq_bvh_build_nodes_device,
trq_scene_rebuild, trq_scene_copy_bvh; DevicePrimitive.build, Scene.rebuild, Scene.bvh).

Leaves made on the GPU must equal the host's trq_bvh_build_nodes_triangles / trq_bvh_build_node byte for byte, NaN, signed
zeros and infinities included; a scene built without leaving the GPU must equal the host-built one; a rebuild must equal
its host restatement (tests/rebuild_util.rebuild_on_host), leave the scene as a fresh trq_scene_create_device of the new tree
would be, trace like port.trace on it, and leave the scene untouched when it fails."""
import ctypes as C

import numpy as np
import pytest

from tracer_b200 import harness as H, layout as L
from tracer_b200._lib import ERR_DEPTH, ERR_INVALID, TrqError, check, lib

from .test_gpu_builder_edges import COMBS
from .test_gpu_parity import assert_like_oracle, gpu_trace
from .test_gpu_tree_shapes import (_check_configurations, _leaf_items, _trace_everything, expected_staging, refit_case, tree_case, tree_rays,
                                   with_finite_tmax)
from .rebuild_util import reachable, rebuild_on_host
from .util import refit_on_host

pytestmark = pytest.mark.gpu
f32 = np.float32


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _dev(a):
    torch = _torch()
    return None if a is None or a.size == 0 else torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()


def _stream():
    return C.c_void_p(_torch().cuda.current_stream().cuda_stream)


def _device_triangle_leaves(tri, idx, base):
    torch = _torch()
    n = idx.size // 3
    out = torch.full((max(n, 1) * 64,), 0xAB, dtype=torch.uint8, device="cuda")
    dt, di = _dev(tri), _dev(idx)
    check(lib.trq_bvh_build_nodes_triangles_device(None if dt is None else dt.data_ptr(), None if di is None else di.data_ptr(), n, base,
                                                   out.data_ptr(), 0, _stream()), "trq_bvh_build_nodes_triangles_device")
    torch.cuda.synchronize()
    return out.cpu().numpy().view(L.bvh_dtype)[:n]


def _host_triangle_leaves(tri, idx, base):
    n = idx.size // 3
    out = np.zeros(n, dtype=L.bvh_dtype)
    if n:
        check(lib.trq_bvh_build_nodes_triangles(tri.ctypes.data, idx.ctypes.data, n, base, out.ctypes.data), "leaves")
    return out


# ----------------------------------------------------------------------------------------------------- 1. device leaves
SPECIAL = np.array([-0.0, 0.0, np.nan, np.inf, -np.inf, 1e-45, -1e-45, 1.1754942e-38, -5.877472e-39, 3.4028235e38, -3.4028235e38,
                    1.0, -1.0, 0.5, -2.0], dtype=f32)


def _special_triangles(seed, n=20000):
    """Vertices drawn from NaN, +-0, +-inf, denormals, +-FLT_MAX and a few ordinary values; every third triangle
    degenerate (a repeated vertex), some with all three the same."""
    rng = np.random.default_rng(seed)
    verts = np.zeros(3000, dtype=L.vertex_dtype)
    verts["v"] = rng.choice(SPECIAL, (verts.size, 3))
    verts["v"][::5] = rng.uniform(-3, 3, (verts[::5].size, 3)).astype(f32)
    idx = rng.integers(0, verts.size, (n, 3)).astype(np.uint32)
    idx[::3, 1] = idx[::3, 0]
    idx[::7, 1:] = idx[::7, :1]
    return verts, idx.reshape(-1)


def _triangle_sets():
    c3_tri, c3_idx = H.cornell_triangle_soup(with_teapot=True, mesh_levels=2, with_coatball=True)
    s_tri = np.zeros(3 * 300_000, dtype=L.vertex_dtype)
    s_idx = np.zeros(3 * 300_000, dtype=np.uint32)
    lib.trqh_make_soup(300_000, 9, f32(0.01), s_tri.ctypes.data, s_idx.ctypes.data)
    sets = {"c3": (c3_tri, c3_idx), "soup": (s_tri, s_idx)}
    for s in (1, 2, 3):
        sets[f"special-s{s}"] = _special_triangles(s)
    sets["one"] = (c3_tri, c3_idx[:3])
    sets["none"] = (c3_tri, c3_idx[:0])
    return sets


def test_device_triangle_leaves_equal_host_leaves(built):
    _torch()
    sets = _triangle_sets()
    assert sets["c3"][1].size // 3 > 1_000_000
    for name, (tri, idx) in sets.items():
        for base in (0, 12345):
            got, want = _device_triangle_leaves(tri, idx, base), _host_triangle_leaves(tri, idx, base)
            assert got.size == idx.size // 3
            bad = np.nonzero(got.view("V64") != want.view("V64"))[0]
            assert bad.size == 0, f"{name} base {base}: {bad.size} leaves differ, first {bad[:3]}: {got[bad[:1]]} vs {want[bad[:1]]}"
    # the special sets reach the boxes: infinities, and components left at FLT_MAX because every corner was NaN
    want = _host_triangle_leaves(*sets["special-s1"], 0)
    assert np.isinf(want["mini"]).any() and (want["mini"] == f32(3.4028235e38)).any()


def _random_models(rng, n):
    """Column-major model matrices: rotations, negative and zero scales, translations, then +-inf / NaN / -0.0 entries."""
    out = np.zeros((n, 16), dtype=f32)
    for k in range(n):
        m = (H.translation4x4(*rng.uniform(-50, 50, 3)) @ H.rotation4x4(float(rng.uniform(0, 6.3)), tuple(rng.normal(size=3)))
             @ H.scale4x4(*rng.choice([-2.0, -1.0, 0.0, 0.5, 1.0, 3.0], 3)))
        out[k] = H.colmajor(m)
    special = rng.random((n, 16)) < 0.08
    out[special] = rng.choice(np.array([np.inf, -np.inf, np.nan, -0.0, 0.0], dtype=f32), special.sum())
    out[::5, 12:15] = -0.0                                           # -0.0 translations: corners land on -0.0 and +0.0
    return out


def _primitive_sets(rng):
    c1 = H.scene_c1().sphereList
    sets = {"cornell-spheres": (L.SPHERE, H.cornell_spheres()), "c1-spheres": (L.SPHERE, c1),
            "cornell-squares": (L.SQUARE, H.cornell_squares()), "cornell-cubes": (L.CUBE, H.cornell_cubes())}
    for name, (p_type, arr) in list(sets.items()):
        r = np.resize(arr, 4000).copy()
        r["model"] = _random_models(rng, r.size)
        boxes = r["box_mini"].copy()
        pick = rng.random(boxes.shape) < 0.05
        boxes[pick] = rng.choice(SPECIAL, pick.sum())
        r["box_mini"] = boxes
        r["model"][1::25] = -0.0                                     # corners land on -0.0 and on +0.0 (ties) ...
        r["box_mini"][1::50], r["box_maxi"][1::50] = -1, 1
        r["box_mini"][26::50], r["box_maxi"][26::50] = 1, 1           # ... or all on -0.0
        sets[name + "-random-models"] = (p_type, r)
    return sets


def test_device_primitive_leaves_equal_host_leaves(built):
    torch = _torch()
    rng = np.random.default_rng(3)
    for name, (p_type, arr) in _primitive_sets(rng).items():
        base = 7 if "random" in name else 0
        want = np.zeros(arr.size, dtype=L.bvh_dtype)
        for k in range(arr.size):
            lo, hi = (np.ascontiguousarray(arr[f][k], dtype=f32) for f in ("box_mini", "box_maxi"))
            m = np.ascontiguousarray(arr["model"][k], dtype=f32)
            check(lib.trq_bvh_build_node(lo.ctypes.data, hi.ctypes.data, m.ctypes.data, p_type, base + k, want[k:k + 1].ctypes.data), "node")
        out = torch.full((arr.size * 64,), 0xCD, dtype=torch.uint8, device="cuda")
        d = _dev(arr)
        check(lib.trq_bvh_build_nodes_device(p_type, d.data_ptr(), arr.size, base, out.data_ptr(), 0, _stream()), "trq_bvh_build_nodes_device")
        got = out.cpu().numpy().view(L.bvh_dtype)
        bad = np.nonzero(got.view("V64") != want.view("V64"))[0]
        assert bad.size == 0, f"{name}: {bad.size} leaves differ, first {bad[:3]}: {got[bad[:1]]} vs {want[bad[:1]]}"
        if "random" in name:                                         # the edge values reach the boxes
            assert (want["mini"].view(np.uint32) == 0x80000000).any() or (want["maxi"].view(np.uint32) == 0x80000000).any(), name
            assert np.isinf(want["maxi"]).any() and (want["maxi"] == -L.FLT_MAX).any(), name


# --------------------------------------------------------------------------------------------- 2. the chain on the device
def _scene_prim(name):
    if name == "c1":
        return H.scene_c1()
    if name == "c2":
        return H.scene_c2()
    if name == "reference_cornell":
        return H.scene_reference_cornell()
    return H.scene_soup(300_000, seed=4, extent=0.004)


def _rays(prim, name, seed=5):
    if name in ("c2", "reference_cornell"):
        return H.cornell_camera_rays(160, 90)
    if name == "c1":
        return H.camera_rays((13, 2, 3), (0, 0, 0), f32(20 * np.pi / 180), 160, 90)
    return H.random_rays(30000, seed=seed)


def _answers(scene, rays):
    return [gpu_trace(scene, rays, any_hit) for any_hit in (False, True)]


def _assert_oracle(port, prim, scene, rays, where):
    for any_hit, got in zip((False, True), _answers(scene, rays)):
        assert_like_oracle(got, port, prim, rays, any_hit, f"{where} any={any_hit}")


@pytest.mark.parametrize("name", ["c1", "c2", "reference_cornell", "soup300k"])
def test_scene_built_on_the_device_equals_the_host_chain(built, port, name):
    _torch()
    from tracer_b200 import DevicePrimitive, Scene
    prim = _scene_prim(name)
    host = Scene(prim, 0)
    dprim = DevicePrimitive.build(_dev(prim.sphereList), _dev(prim.squareList), _dev(prim.cubeList), _dev(prim.triList), _dev(prim.idxList))
    dev = Scene(dprim, 0)
    assert dev.bvh().tobytes() == host.bvh().tobytes() == prim.bvhList.tobytes(), name
    assert dev.info == host.info, name
    rays = _rays(prim, name)
    for a, b in zip(_answers(host, rays), _answers(dev, rays)):
        assert a.tobytes() == b.tobytes(), name
    _assert_oracle(port, prim, dev, rays, name)


@pytest.mark.parametrize("name", ["c1", "c2", "reference_cornell"])
def test_rebuild_of_an_unchanged_scene_is_the_identity(built, port, name):
    _torch()
    from tracer_b200 import Scene
    prim = _scene_prim(name)
    scene = Scene(prim, 0)
    rays = _rays(prim, name)
    before, info = _answers(scene, rays), dict(scene.info)
    scene.rebuild()
    assert scene.bvh().tobytes() == prim.bvhList.tobytes() and scene.info == info, name
    for a, b in zip(before, _answers(scene, rays)):
        assert a.tobytes() == b.tobytes(), name


# ------------------------------------------------------------------------------------------------ 4. rebuild after motion
def _moved(prim, how, rng):
    v = prim.triList.copy()
    if how == "jitter":
        v["v"] += rng.uniform(-0.002, 0.002, v["v"].shape).astype(f32)
    else:                                                            # every triangle takes another one's place
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
def test_rebuild_after_motion(built, port, how, source):
    torch = _torch()
    from tracer_b200 import Scene
    rng = np.random.default_rng(len(how) + len(source))
    prim = H.scene_soup(20000, seed=6, extent=0.01)
    verts = _moved(prim, how, rng)
    want = rebuild_on_host(prim, verts)
    scene = Scene(prim, 0)
    scene.rebuild(verts if source == "host" else torch.from_numpy(verts.view(np.uint8).reshape(-1).copy()).cuda())
    assert scene.bvh().tobytes() == want.bvhList.tobytes()
    assert scene.info == _fresh_info(want)
    cfgs = _check_configurations(scene, f"rebuild {how} {source}")
    rays = H.random_rays(6000, seed=11)
    rays_any = with_finite_tmax(rng, rays, _leaf_items(want))
    _trace_everything(port, want, scene, rays, rays_any, f"rebuild {how} ({source} vertices)", cfgs)
    # a refit of the rebuilt tree still follows the vertices
    again = verts.copy()
    again["v"] += rng.uniform(-0.003, 0.003, again["v"].shape).astype(f32)
    scene.update_vertices(again)
    refit = refit_on_host(want, again)
    assert scene.bvh().tobytes() == refit.bvhList.tobytes()
    _assert_oracle(port, refit, scene, rays, f"refit after rebuild {how} ({source})")
    scene.close()


# ------------------------------------------------------------------------------------------- 5. caller-built host trees
CALLER = ["split-random-inf-odd", "split-bfs-inflated-mixed", "split-random-nonnest-lattice", "combLnear-post-tight",
          "spine-random-tight", "unreachable", "one_leaf", "two_leaves"]


@pytest.mark.parametrize("name", CALLER)
def test_rebuild_of_caller_built_trees(built, port, name):
    _torch()
    from tracer_b200 import Scene
    rng = np.random.default_rng(sum(map(ord, name)))
    if name in ("unreachable", "one_leaf", "two_leaves"):
        prim, verts = refit_case(name)
    else:
        prim = tree_case(name)[0]
        verts = prim.triList.copy()
        verts["v"] += rng.uniform(-0.05, 0.05, verts["v"].shape).astype(f32)
    want = rebuild_on_host(prim, verts, gpu=0)          # the GPU builder's tree (sorted fallback nodes: include/tracer_rq.h)
    scene = Scene(prim, 0)
    scene.rebuild(verts)
    got = scene.bvh()
    assert got.tobytes() == want.bvhList.tobytes(), name
    n_leaf = int(((prim.bvhList["pType"] != L.BVH) & reachable(prim.bvhList)).sum())
    assert scene.info["nNode"] == got.size == 2 * n_leaf - 1, name
    assert scene.info == _fresh_info(want), name
    if scene.info["nInterior"]:
        cfgs = _check_configurations(scene, name)
    else:                                                # a lone leaf has no top-of-tree block to stage
        cfgs = [c for c, cfg in enumerate(Scene.kernel_configs()) if expected_staging(cfg, 0, 0)[0]]
        assert cfgs == [0] and scene.kernel_config() == Scene.kernel_configs()[0]
    lv = _leaf_items(want)
    rays = tree_rays(rng, want, lv, n=2000)
    _trace_everything(port, want, scene, rays, with_finite_tmax(rng, rays, lv), f"rebuild {name}", cfgs)
    scene.close()


# ---------------------------------------------------------------------------------------- 6. a failed rebuild changes nothing
def test_failed_rebuild_leaves_the_scene_intact(built, port):
    _torch()
    from tracer_b200 import Scene
    base, lo, hi = COMBS[35]
    x = np.array([float(base) ** k for k in range(lo, hi + 1)]).astype(f32)
    prim = H.scene_soup(x.size, seed=2, extent=0.05)
    comb = prim.triList.copy()                           # triangle i flat at x = 11^perm(i), spanning [0, 1] in y and z
    corners = np.array([[0, 0, 0], [0, 1, 0], [0, 0, 1]], dtype=f32)
    comb["v"] = np.tile(corners, (x.size, 1))
    comb["v"][:, 0] = np.repeat(x[np.random.default_rng(1).permutation(x.size)], 3)
    with pytest.raises(TrqError) as e:
        rebuild_on_host(prim, comb)
    assert e.value.status == ERR_DEPTH
    scene = Scene(prim, 0)
    rays = H.random_rays(5000, seed=3)
    bvh, info, before = scene.bvh().tobytes(), dict(scene.info), _answers(scene, rays)
    with pytest.raises(TrqError) as e:
        scene.rebuild(comb)
    assert e.value.status == ERR_DEPTH and "35" in str(e.value), str(e.value)
    assert lib.trq_scene_rebuild(scene._h, comb.ctypes.data, comb.size - 1, L.HOST_PTRS) == ERR_INVALID   # not the scene's count
    assert b"vertices" in lib.trq_last_error_string()
    assert scene.bvh().tobytes() == bvh and scene.info == info
    for a, b in zip(before, _answers(scene, rays)):
        assert a.tobytes() == b.tobytes()
    scene.rebuild()                                      # the scene's vertices are the old ones: the same tree again
    assert scene.bvh().tobytes() == bvh and scene.info == info
    _assert_oracle(port, prim, scene, rays, "after a failed rebuild")


# ---------------------------------------------------------------------------------------------- 7. configuration bookkeeping
def test_rebuild_redoes_the_configurations(built):
    """comb31 (maxDepth 31, a long far-child stack per ray) rebuilt into a shallow tree: each configuration's usability and
    staged count become a fresh scene's; without a caller's choice the automatic one is taken, a caller's choice stays."""
    _torch()
    from tracer_b200 import DevicePrimitive, Scene
    prim, verts = refit_case("comb31")
    want = rebuild_on_host(prim, verts, gpu=0)
    names = Scene.kernel_configs()
    fresh = Scene(DevicePrimitive.from_host(want, "cuda:0"), 0)
    staged = {}
    for c in range(len(names)):
        try:
            staged[c] = fresh.set_kernel_config(c)
        except TrqError:
            staged[c] = None
    fresh.set_kernel_config(-1)
    for chosen in (None, 0):
        scene = Scene(prim, 0)
        assert scene.info["maxDepth"] == 31
        if chosen is not None:
            scene.set_kernel_config(chosen)
        scene.rebuild(verts)
        assert scene.info["maxDepth"] < 31 and scene.info == fresh.info
        assert scene.kernel_config() == (fresh.kernel_config() if chosen is None else names[chosen])
        current = scene.kernel_config()
        for c in range(len(names)):
            if staged[c] is None:
                with pytest.raises(TrqError):
                    scene.set_kernel_config(c)
            else:
                assert scene.set_kernel_config(c) == staged[c], (chosen, names[c])
        assert current == names[0] or chosen is None
        _check_configurations(scene, f"comb31 rebuilt, chosen {chosen}")
        scene.close()
    fresh.close()


# -------------------------------------------------------------------------------------------------------------- 8. ordering
def test_rebuild_waits_for_traces_in_flight(built):
    """A large trace queued on a side stream just before a rebuild returns the answers of the tree before it."""
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
    scene.rebuild(moved)
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    after = scene.hit(rays)
    torch.cuda.synchronize()
    assert not torch.equal(after, want)                  # the rebuild took effect for the next trace
    scene.close()
