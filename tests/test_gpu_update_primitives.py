"""trq_scene_update_primitives / Scene.update_primitives: moving spheres, squares, cubes and vertices of a live scene.

After every update the scene's node array must equal the host restatement (tests/update_util.update_on_host) byte for
byte, its info must be unchanged, it must trace like port.trace on the new lists and the restated tree (every usable
configuration, the reference-layout kernel, 16-byte hits, trq_expand_hits), and like a scene created afresh from them.
A failed update must leave the scene as it was."""
import ctypes as C

import numpy as np
import pytest

from tracer_b200 import harness as H, layout as L
from tracer_b200._lib import ERR_INVALID, SceneDesc, TrqError, lib
from tracer_b200.scene import Primitive

from .rebuild_util import rebuild_on_host
from .test_gpu_rebuild import _assert_oracle, _dev, _primitive_sets, _random_models
from .test_gpu_tree_shapes import (Leaves, Topo, _info, _leaf_items, _trace_everything, boxes, comb, expected_staging, make_prim,
                                   numbering, tree_case, tree_rays, with_finite_tmax)
from .update_util import depths, primitive_leaves, update_on_host

pytestmark = pytest.mark.gpu
f32 = np.float32


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


# ------------------------------------------------------------------------------------------------------------- helpers
def _update(scene, source, spheres=None, squares=None, cubes=None, triList=None):
    lists = dict(spheres=spheres, squares=squares, cubes=cubes, triList=triList)
    lists = {k: (v if source == "host" else _dev(v)) for k, v in lists.items() if v is not None}
    scene.update_primitives(**lists)


def _cfgs(scene):
    from tracer_b200 import Scene
    info = _info(scene)
    return [c for c, cfg in enumerate(Scene.kernel_configs()) if expected_staging(cfg, info["maxDepth"], info["topNodes"])[0]]


def _hits(scene, rays, rays_any, cfgs):
    """Packed-kernel hits in the order _trace_everything returns them."""
    from tracer_b200 import rays_to_torch
    out = []
    for any_hit, r in ((False, rays), (True, rays_any)):
        d = rays_to_torch(r, f"cuda:{scene.device}")
        for c in cfgs:
            scene.set_kernel_config(c)
            out.append(scene.hit(d, any=any_hit).cpu().numpy().view(L.hit_dtype).reshape(-1))
        scene.set_kernel_config(-1)
    return out


def _same_except_boxes(a, b, where):
    for k in L.bvh_dtype.names:
        if k not in ("mini", "maxi"):
            assert a[k].tobytes() == b[k].tobytes(), f"{where}: {k}"


def _check(port, scene, want, info, rays, rays_any, where, exact=True):
    """The updated scene against the restatement `want`. exact=False (non-finite records): leaves byte for byte, interior
    boxes by value (+-0 equal, NaN equal), every other field byte for byte; the traces then run on the scene's own tree and
    are compared with a scene created from it, not with the oracle."""
    from tracer_b200 import Scene
    got = scene.bvh()
    if exact:
        assert got.tobytes() == want.bvhList.tobytes(), f"{where}: node array"
    else:
        w = want.bvhList
        _same_except_boxes(got, w, where)
        leaf = got["pType"] != L.BVH
        assert got[leaf].tobytes() == w[leaf].tobytes(), f"{where}: leaves"
        for k in ("mini", "maxi"):
            assert np.array_equal(got[k][~leaf], w[k][~leaf], equal_nan=True), f"{where}: interior {k}"
        want = Primitive(**{**want.__dict__, "bvhList": got})
    assert _info(scene) == info, where
    cfgs = _cfgs(scene)
    if exact:
        _trace_everything(port, want, scene, rays, rays_any, where, cfgs)
    fresh = Scene(want, 0)
    for a, b in zip(_hits(scene, rays, rays_any, cfgs), _hits(fresh, rays, rays_any, cfgs)):
        assert a.tobytes() == b.tobytes(), f"{where}: a scene created from the new lists traces differently"
    fresh.close()


def _moved_spheres(s, rng, d, lift=None):
    s = s.copy()
    off = rng.uniform(-d, d, (s.size, 3)).astype(f32) if lift is None else lift
    s["center"] += off
    s["box_mini"] += off
    s["box_maxi"] += off
    return s


def _moved_squares(s, rng, d):
    s = s.copy()
    n = np.arange(s.size)
    k = s["axis_k"].astype(np.int64)
    dk = rng.uniform(-d, d, s.size).astype(f32)
    s["value_k"] += dk
    s["box_mini"][n, k] += dk
    s["box_maxi"][n, k] += dk
    i = s["axis_i"].astype(np.int64)
    di = rng.uniform(-d, d, s.size).astype(f32)
    s["range_i"] += di[:, None]
    s["box_mini"][n, i] += di
    s["box_maxi"][n, i] += di
    return s


def _reposed_cubes(c, rng, d, scale):
    out = c.copy()
    for k in range(c.size):
        t = c["model"][k][12:15] + rng.uniform(-d, d, 3).astype(f32)
        m = H.translation4x4(*t) @ H.rotation4x4(float(rng.uniform(0, 6.3)), tuple(rng.normal(size=3))) @ H.scale4x4(*rng.uniform(0.5, 1.5, 3) * scale)
        out[k] = H.make_cube(m, int(c["material"][k]))
        out[k]["box_mini"], out[k]["box_maxi"] = c["box_mini"][k], c["box_maxi"][k]
    return out


def _jittered(v, rng, d):
    v = v.copy()
    v["v"] += rng.uniform(-d, d, v["v"].shape).astype(f32)
    return v


def _rays_for(rng, prim, n=2000):
    lv = _leaf_items(prim)
    rays = tree_rays(rng, prim, lv, n=n)
    return rays, with_finite_tmax(rng, rays, lv)


# ----------------------------------------------------------------------------------------------------------------- C1
def _c1_rays(rng):
    rays = np.concatenate([H.camera_rays((13, 2, 3), (0, 0, 0), f32(20 * np.pi / 180), 160, 90),
                           H.camera_rays((-12, 2.5, -4), (0, 0.5, 0), f32(30 * np.pi / 180), 96, 54)])
    lv = _leaf_items(H.scene_c1())
    return rays, with_finite_tmax(rng, rays, lv)


@pytest.mark.parametrize("source", ["host", "device"])
def test_c1_spheres_move(built, port, source):
    _torch()
    from tracer_b200 import Scene
    rng = np.random.default_rng(11 if source == "host" else 12)
    prim = H.scene_c1()
    rays, rays_any = _c1_rays(rng)
    scene = Scene(prim, 0)
    info = _info(scene)
    before = _hits(scene, rays, rays_any, _cfgs(scene))
    moved = _moved_spheres(prim.sphereList, rng, 0.4)
    _update(scene, source, spheres=moved)
    _check(port, scene, update_on_host(prim, spheres=moved), info, rays, rays_any, f"c1 all moved ({source})")
    # a MovingSphere at t = 1: only the small spheres, lifted
    lifted = prim.sphereList.copy()
    small = lifted["radius"] == f32(0.2)
    assert small.sum() == 438
    lift = np.zeros((lifted.size, 3), dtype=f32)
    lift[small, 1] = rng.uniform(0, 0.5, small.sum()).astype(f32)
    lifted = _moved_spheres(lifted, rng, 0, lift=lift)
    _update(scene, source, spheres=lifted)
    _check(port, scene, update_on_host(prim, spheres=lifted), info, rays, rays_any, f"c1 small lifted ({source})")
    # and back: the original answers return
    _update(scene, source, spheres=prim.sphereList)
    assert scene.bvh().tobytes() == prim.bvhList.tobytes() and _info(scene) == info
    for a, b in zip(before, _hits(scene, rays, rays_any, _cfgs(scene))):
        assert a.tobytes() == b.tobytes(), "c1 back"
    scene.close()


# ---------------------------------------------------------------------------------------------- reference Cornell mix
@pytest.mark.parametrize("source", ["host", "device"])
def test_reference_cornell_everything_moves(built, port, source):
    _torch()
    from tracer_b200 import Scene
    rng = np.random.default_rng(21 if source == "host" else 22)
    prim = H.scene_reference_cornell()
    scene = Scene(prim, 0)
    info = _info(scene)
    sph = _moved_spheres(prim.sphereList, rng, 20)
    sq = _moved_squares(prim.squareList, rng, 5)
    cubes = _reposed_cubes(prim.cubeList, rng, 40, 150)
    verts = _jittered(prim.triList, rng, 1.5)
    _update(scene, source, spheres=sph, squares=sq, cubes=cubes, triList=verts)
    want = update_on_host(prim, spheres=sph, squares=sq, cubes=cubes, verts=verts)
    rays, rays_any = _rays_for(rng, want)
    rays = np.concatenate([H.cornell_camera_rays(160, 90), rays])
    rays_any = np.concatenate([with_finite_tmax(rng, H.cornell_camera_rays(160, 90), _leaf_items(want)), rays_any])
    _check(port, scene, want, info, rays, rays_any, f"reference cornell ({source})")
    # a cube with a down-scaling model matrix (test_gpu_producers.test_cube_with_a_down_scaling_model_matrix), rays inside it
    model = H.translation4x4(0.5, -0.25, 2.0) @ H.rotation4x4(0.3, (0, 1, 0)) @ H.scale4x4(0.01, 0.02, 0.015)
    c = H.make_cube(model, 3)
    c["box_mini"], c["box_maxi"] = (-100, -60, -80), (100, 60, 80)
    down = np.array([c, H.cornell_cubes()[0]], dtype=L.cube_dtype)
    _update(scene, source, cubes=down)
    want = update_on_host(want, cubes=down)
    n = 3000
    inside = np.zeros(n, dtype=L.ray_dtype)
    local = rng.uniform([-95, -55, -75], [95, 55, 75], size=(n, 3))
    M = model.astype(np.float64)
    inside["o"] = ((M[:3, :3] @ local.T).T + M[:3, 3]).astype(f32)
    dd = rng.normal(size=(n, 3))
    inside["d"] = (dd / np.linalg.norm(dd, axis=1, keepdims=True)).astype(f32)
    inside["tmax"] = rng.uniform(0.5, 150.0, size=n).astype(f32)
    _check(port, scene, want, info, inside, inside, f"reference cornell down-scaling cube ({source})")
    scene.close()


# ------------------------------------------------------------------------------------------------ caller-built trees
def _small(kind, n):
    lv = Leaves()
    if kind == "sphere":
        lv.sphere(0.5, (0, 0, 0))
    else:
        lv.square(0, (-1, 1), 2, (-1, 1), 1, 0)
        lv.square(0, (0, 2), 1, (0, 2), 2, 1)
    t = Topo()
    t.root = t.add(leaf=0) if n == 1 else t.add(t.add(leaf=0), t.add(leaf=1))
    lo, hi = boxes(t, lv, "tight", None)
    perm = np.zeros(1, dtype=np.int64) if n == 1 else np.array([2, 1, 0])
    return make_prim(t, lv, perm, lo, hi)


def _sphere_comb():
    """A depth-31 comb of sphere leaves in random numbering."""
    lv = Leaves()
    for k in range(33):
        lv.sphere(0.45, (f32(100 - k), 0, 0))
    t = comb(31, True)
    perm = numbering(t, "random", np.random.default_rng(4))
    lo, hi = boxes(t, lv, "tight", None)
    return make_prim(t, lv, perm, lo, hi)


def _with_orphan_primitives(prim, rng):
    """Appends sphere, square and cube leaves the root does not reach (valid pIndex, parent naming a reachable interior
    node, a box of their own): an update must not touch them."""
    b = prim.bvhList
    inner = np.nonzero(b["pType"] == L.BVH)[0]
    orphans = np.zeros(12, dtype=L.bvh_dtype)
    orphans["pType"] = np.tile([L.SPHERE, L.SQUARE, L.CUBE], 4)
    for k, t in enumerate(orphans["pType"]):
        n = {L.SPHERE: prim.sphereList.size, L.SQUARE: prim.squareList.size, L.CUBE: prim.cubeList.size}[int(t)]
        orphans["pIndex"][k] = rng.integers(0, n)
    orphans["parent"] = rng.choice(inner, orphans.size)
    orphans["mini"], orphans["maxi"] = f32(-1234.5), f32(2345.25)
    return Primitive(**{**prim.__dict__, "bvhList": np.concatenate([b, orphans])})


CALLER = ["split-random-inflated-mixed", "split-random-inf-odd", "comb31-spheres", "one_leaf_sphere", "two_leaf_square", "unreachable"]


def _caller_case(name):
    if name == "comb31-spheres":
        return _sphere_comb()
    if name == "one_leaf_sphere":
        return _small("sphere", 1)
    if name == "two_leaf_square":
        return _small("square", 2)
    if name == "unreachable":
        return _with_orphan_primitives(tree_case("split-random-inflated-mixed")[0], np.random.default_rng(9))
    return tree_case(name)[0]


@pytest.mark.parametrize("name", CALLER)
def test_caller_built_trees(built, port, name):
    _torch()
    from tracer_b200 import Scene
    rng = np.random.default_rng(sum(map(ord, name)))
    source = "device" if CALLER.index(name) % 2 else "host"
    prim = _caller_case(name)
    scene = Scene(prim, 0)
    info = _info(scene)
    lists = dict(spheres=_moved_spheres(prim.sphereList, rng, 0.3) if prim.sphereList.size else None,
                 squares=_moved_squares(prim.squareList, rng, 0.3) if prim.squareList.size else None,
                 cubes=_reposed_cubes(prim.cubeList, rng, 0.3, 0.5) if prim.cubeList.size else None,
                 triList=_jittered(prim.triList, rng, 0.1) if prim.triList.size else None)
    _update(scene, source, **lists)
    want = update_on_host(prim, lists["spheres"], lists["squares"], lists["cubes"], lists["triList"])
    rays, rays_any = _rays_for(rng, want)
    if name == "comb31-spheres":
        assert info["maxDepth"] == 31
    _check(port, scene, want, info, rays, rays_any, f"{name} ({source})")
    got = scene.bvh()
    unreached = depths(got) < 0
    keep = unreached | ~np.isin(got["pType"], [L.BVH, L.SPHERE, L.SQUARE, L.CUBE, L.TRIANGLE])
    assert got[keep].tobytes() == prim.bvhList[keep].tobytes(), f"{name}: unreachable or unknown leaves changed"
    if name == "unreachable":
        assert unreached.sum() == 12
    if name in ("one_leaf_sphere", "two_leaf_square"):
        assert got["mini"][0].tobytes() != prim.bvhList["mini"][0].tobytes()
    scene.close()


# ------------------------------------------------------------------------------------------------ adversarial records
def test_adversarial_records(built, port):
    """Records with NaN, +-inf, -0.0, denormals and +-FLT_MAX in their matrices and boxes: every leaf is trq_bvh_build_node
    of its record byte for byte."""
    _torch()
    from tracer_b200 import Scene
    rng = np.random.default_rng(3)
    sets = _primitive_sets(rng)
    sph, sq, cubes = (sets[k][1] for k in ("c1-spheres-random-models", "cornell-squares-random-models", "cornell-cubes-random-models"))
    sane = [np.resize(a, 4000).copy() for a in (H.scene_c1().sphereList, H.cornell_squares(), H.cornell_cubes())]
    prim = H.build_primitive(spheres=sane[0], squares=sane[1], cubes=sane[2])
    scene = Scene(prim, 0)
    info = _info(scene)
    for k, source in enumerate(("host", "device")):
        lists = dict(spheres=sph, squares=sq, cubes=cubes)
        if k:
            lists = {n: a.copy() for n, a in lists.items()}
            for a in lists.values():
                a["model"] = _random_models(rng, a.size)
        _update(scene, source, **lists)
        want = update_on_host(prim, **lists)
        got = scene.bvh()
        for t, key in ((L.SPHERE, "spheres"), (L.SQUARE, "squares"), (L.CUBE, "cubes")):
            at = np.nonzero(got["pType"] == t)[0]
            made = primitive_leaves(lists[key], t)[got["pIndex"][at]]
            for f in ("mini", "maxi"):
                assert got[f][at].tobytes() == made[f].tobytes(), (source, key, f)
        assert np.isnan(got["mini"]).any() or np.isinf(got["maxi"]).any()
        rays, rays_any = _rays_for(rng, prim)
        _check(port, scene, want, info, rays, rays_any, f"adversarial ({source})", exact=False)
    scene.close()


# ------------------------------------------------------------------------------------------------------------------ C4
def test_c4_spheres_and_lights_move(built, port):
    torch = _torch()
    from tracer_b200 import Scene
    rng = np.random.default_rng(4)
    prim = H.scene_c4(levels=0)
    assert prim.nTri == 62558 and prim.sphereList.size == 10012
    scene = Scene(prim, 0)
    info = _info(scene)
    sph = _moved_spheres(prim.sphereList, rng, 3)
    _update(scene, "device", spheres=sph)
    want = update_on_host(prim, spheres=sph)
    cam = H.cornell_camera_rays(96, 54)
    rays = np.concatenate([cam, H.random_rays(3000, seed=8, lo=(-245, 0, 0), hi=(800, 555, 555))])
    rays_any = with_finite_tmax(rng, rays, _leaf_items(want))
    _check(port, scene, want, info, rays, rays_any, "c4 spheres moved")
    # the lights: squareList has no leaves here, so the node array stays as it is, and the shadow rays follow the lights
    bvh = scene.bvh().tobytes()
    sq = prim.squareList.copy()
    sq[5] = H.make_square(0, (300, 455), 2, (100, 255), 1, 554.9, int(sq["material"][5]))
    sq[6] = H.make_square(1, (250, 350), 2, (150, 250), 0, -280, int(sq["material"][6]))
    _update(scene, "host", squares=sq)
    assert scene.bvh().tobytes() == bvh and _info(scene) == info
    d = scene.cast_rays((278, 278, -800), (278, 278, 278), (0, 1, 0), f32(45 * (np.pi / 180)), 320, 180)
    hits = scene.hit(d)
    recs = scene.expand(d, hits).cpu().numpy().view(L.record_dtype).reshape(-1)
    out, src, cnt = scene.spawn_shadow(d, hits, 5, 6, seed_base=11)
    want_rays, wsrc = H.shadow_rays(recs, sq[5:6], sq[6:7], seed_base=11)
    old_rays, _ = H.shadow_rays(recs, prim.squareList[5:6], prim.squareList[6:7], seed_base=11)
    n = int(cnt.item())
    assert n == want_rays.size == int(recs["hit"].sum()) > 0
    order = np.argsort(src.cpu().numpy()[:n].astype(np.uint32), kind="stable")
    got = out.cpu().numpy().view(L.ray_dtype).reshape(-1)[:n][order]
    assert np.array_equal(src.cpu().numpy()[:n].astype(np.uint32)[order], wsrc)
    assert np.array_equal(got["o"].view(np.uint32), want_rays["o"].view(np.uint32))
    assert np.array_equal(got["d"].view(np.uint32), want_rays["d"].view(np.uint32)), "shadow directions use no libm: bit-exact"
    assert np.array_equal(got["tmax"].view(np.uint32), want_rays["tmax"].view(np.uint32)), "shadow lengths: strict fp32 sqrtf, bit-exact"
    assert not np.array_equal(want_rays["d"], old_rays["d"])
    torch.cuda.synchronize()
    scene.close()


# ------------------------------------------------------------------------------------------------------- triList only
def test_trilist_only_equals_update_vertices(built, port):
    _torch()
    from tracer_b200 import Scene
    rng = np.random.default_rng(5)
    prim = H.scene_reference_cornell()
    verts = _jittered(prim.triList, rng, 2.0)
    a, b = Scene(prim, 0), Scene(prim, 0)
    a.update_primitives(triList=verts)
    b.update_vertices(verts)
    assert a.bvh().tobytes() == b.bvh().tobytes() == update_on_host(prim, verts=verts).bvhList.tobytes()
    rays, rays_any = _rays_for(rng, update_on_host(prim, verts=verts))
    for x, y in zip(_hits(a, rays, rays_any, _cfgs(a)), _hits(b, rays, rays_any, _cfgs(b))):
        assert x.tobytes() == y.tobytes()
    a.close(); b.close()


# -------------------------------------------------------------------------------------------------- update, then rebuild
@pytest.mark.parametrize("name", ["c1", "reference_cornell"])
def test_update_then_rebuild(built, port, name):
    _torch()
    from tracer_b200 import Scene
    rng = np.random.default_rng(6)
    prim = H.scene_c1() if name == "c1" else H.scene_reference_cornell()
    sph = _moved_spheres(prim.sphereList, rng, 0.6 if name == "c1" else 60)
    scene = Scene(prim, 0)
    scene.update_primitives(spheres=sph)
    scene.rebuild()
    want = rebuild_on_host(update_on_host(prim, spheres=sph), gpu=0)
    assert scene.bvh().tobytes() == want.bvhList.tobytes(), name
    assert scene.bvh().tobytes() != prim.bvhList.tobytes(), name
    rays = _c1_rays(rng)[0] if name == "c1" else H.cornell_camera_rays(160, 90)
    _assert_oracle(port, want, scene, rays, f"{name} update then rebuild")
    scene.close()


# ------------------------------------------------------------------------------------------- a failed update changes nothing
def test_failed_update_leaves_the_scene_intact(built, port):
    _torch()
    from tracer_b200 import Scene, rays_to_torch
    prim = H.scene_reference_cornell()
    scene = Scene(prim, 0)
    rng = np.random.default_rng(7)
    rays, rays_any = _rays_for(rng, prim, n=1000)
    bvh, info, before = scene.bvh().tobytes(), _info(scene), _hits(scene, rays, rays_any, _cfgs(scene))
    d = rays_to_torch(rays, "cuda:0")
    recs = scene.expand(d, scene.hit(d)).cpu().numpy()
    moved = _moved_spheres(prim.sphereList, rng, 30)
    with pytest.raises(TrqError) as e:
        scene.update_primitives(spheres=moved[:-1], squares=_moved_squares(prim.squareList, rng, 5))
    assert e.value.status == ERR_INVALID and "spheres" in str(e.value)
    with pytest.raises(TypeError):
        scene.update_primitives(spheres=moved, squares=_dev(prim.squareList))
    desc = SceneDesc()
    desc.sphereList, desc.nSphere = moved.ctypes.data, moved.size
    desc.idxList, desc.nTri = prim.idxList.ctypes.data, prim.nTri
    assert lib.trq_scene_update_primitives(scene._h, C.byref(desc), L.HOST_PTRS) == ERR_INVALID
    desc = SceneDesc()
    desc.sphereList, desc.nSphere = moved.ctypes.data, moved.size
    desc.nCube = prim.cubeList.size
    assert lib.trq_scene_update_primitives(scene._h, C.byref(desc), L.HOST_PTRS) == ERR_INVALID
    assert b"NULL array" in lib.trq_last_error_string()
    assert scene.bvh().tobytes() == bvh and _info(scene) == info
    for a, b in zip(before, _hits(scene, rays, rays_any, _cfgs(scene))):
        assert a.tobytes() == b.tobytes()
    assert scene.expand(d, scene.hit(d)).cpu().numpy().tobytes() == recs.tobytes()
    _assert_oracle(port, prim, scene, rays, "after failed updates")
    scene.close()


# ---------------------------------------------------------------------------------------------------------------- ordering
def test_update_waits_for_traces_in_flight(built):
    """A large trace queued on a side stream just before an update returns the answers of the scene before it."""
    torch = _torch()
    from tracer_b200 import Scene, rays_to_torch
    prim = H.scene_c1()
    scene = Scene(prim, 0)
    rays = rays_to_torch(H.random_rays(1 << 22, seed=4, lo=(-11, 0, -11), hi=(11, 2, 11)), "cuda:0")
    want = scene.hit(rays)
    torch.cuda.synchronize()
    moved = _moved_spheres(prim.sphereList, np.random.default_rng(2), 0.5)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        got = scene.hit(rays, stream=side.cuda_stream)
    scene.update_primitives(spheres=moved)
    torch.cuda.synchronize()
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))         # bits: a sphere hit's u, v may be NaN
    after = scene.hit(rays)
    torch.cuda.synchronize()
    assert not torch.equal(after.view(torch.int32), want.view(torch.int32))                  # the update took effect for the next trace
    scene.close()
