"""GPU: special-valued rays through every trace path, degenerate surfaces through trq_expand_hits and the spawns, and the
libm-dependent values (sphere uv, bounce directions) checked exactly against float64.

Rules: ids, flags and t bit for bit; u / v bit for bit except on sphere hits; where the oracle's float is NaN, NaN-ness only.
Sphere uv and bounce directions depend on libm only through atan2f / asinf and cosf / sinf, so they are checked against every
float32 value within the CUDA Math API's documented maximum error of the float64 result, pushed through the rest of the
float32 chain in numpy: the device's bits must be one of those outcomes. Generators: tests/test_special_rays_cpu.py."""
import os

import numpy as np
import pytest

from tracer_b200 import layout as L

from .test_gpu_fuzz import _assert_records
from .test_gpu_parity import _torch, gpu_trace
from .test_special_rays_cpu import (_nan_aware_equal, _seen, aimed_rays, assert_sphere_uv, bounce_direction_candidates, comb_right,
                                    degenerate_scene, flat_cube_scene, nan_origin_rays, one_leaf, pole_spheres_scene, special_rays)
from .util import bits

pytestmark = pytest.mark.gpu

f32 = np.float32


def assert_hits_exact(got, want, where, records=None):
    """trq_hit against the oracle: ids and flags equal, t bit for bit, u / v bit for bit except sphere hits (NaN-aware);
    sphere uv by assert_sphere_uv against the oracle's records, which are required when the oracle reports a sphere hit."""
    assert got.size == want.size
    for k in ("flags", "pType", "pIndex", "leafNode", "material"):
        bad = np.nonzero(got[k] != want[k])[0]
        assert bad.size == 0, f"{where}: {k} differs on {bad.size} rays, first {bad[:5]}: got {got[k][bad[:5]]} want {want[k][bad[:5]]}"
    assert _nan_aware_equal(got["t"], want["t"]), f"{where}: t"
    hit = (want["flags"] & 1) == 1
    sph = hit & (want["pType"] == L.SPHERE)
    for k in ("u", "v"):
        assert _nan_aware_equal(got[k][hit & ~sph], want[k][hit & ~sph]), f"{where}: {k}"
    if sph.any():
        assert records is not None, f"{where}: {int(sph.sum())} sphere hits: pass the oracle's records to check their uv"
        assert records.size == want.size, f"{where}: records of other rays"
        assert_sphere_uv(got["u"][sph], got["v"][sph], records["gn"][sph], want["u"][sph], want["v"][sph], where)


def assert_records_exact(scene, rays, hits_dev, want, where):
    """trq_expand_hits: every HitRecord field NaN-aware bit for bit (_assert_records), and sphere uv exactly."""
    from tracer_b200 import rays_to_torch
    _assert_records(scene, rays, hits_dev, want, where)
    recs = scene.expand(rays_to_torch(rays, f"cuda:{scene.device}"), hits_dev).cpu().numpy().view(L.record_dtype).reshape(-1)
    w = want["records"]
    sph = (w["hit"] == 1) & (want["hits"]["pType"] == L.SPHERE)
    if sph.any():
        assert_sphere_uv(recs["uv"][sph, 0], recs["uv"][sph, 1], w["gn"][sph], w["uv"][sph, 0], w["uv"][sph, 1], where + " expand")
    return recs


def assert_bounce_directions(dirs, sn, src, seed_base, where, uu=None):
    """Each device direction equals one candidate of bounce_direction_candidates, component bits NaN-aware. uu: the two
    draws of each ray, by default those of PCG32(seed_base + src, 1)."""
    from tracer_b200 import harness as H
    if uu is None:
        uu = np.stack([H.pcg32_floats(seed_base + int(i), 1, 2) for i in src])
    cand = bounce_direction_candidates(sn, uu[:, 0], uu[:, 1])
    nan_ok = np.isnan(cand) & np.isnan(dirs)[:, None, :]
    same = (bits(cand) == bits(dirs)[:, None, :]) | nan_ok
    ok = same.all(axis=2).any(axis=1)
    bad = np.nonzero(~ok)[0]
    assert bad.size == 0, f"{where}: {bad.size} bounce directions match no candidate, first {bad[:3]}: {dirs[bad[:3]]}, sn {sn[bad[:3]]}"


# ----------------------------------------------------------------------------------------------------------- scenes
def _trace_scenes(rng):
    from tracer_b200 import harness as H
    yield "cornell mixed", H.scene_reference_cornell(), 20000, 64
    yield "soup", H.scene_soup(3000, seed=int(rng.integers(1 << 30)), extent=0.15), 20000, 64
    sph = np.array([H.make_sphere(float(rng.uniform(0.2, 1.5)), rng.uniform(-3, 3, 3), i) for i in range(60)], dtype=L.sphere_dtype)
    yield "spheres", H.build_primitive(spheres=sph), 20000, 64
    yield "one leaf", one_leaf(), 4000, 256
    yield "comb31", comb_right(), 4000, 256
    yield "degenerate", degenerate_scene()[0], 8000, 64


def _check_all_paths(port, prim, rays, where):
    """Reference-layout kernel, every packed configuration with trq_hit and trq_hit16, sort=True, trq_trace_indirect, the
    host-pointer path in small chunks, and trq_expand_hits: all against the oracle."""
    torch = _torch()
    from tracer_b200 import Scene, hits_to_numpy, rays_to_torch
    scene = Scene(prim, 0)
    d = rays_to_torch(rays, "cuda:0")
    n = rays.size
    for any_hit in (False, True):
        want = port.trace(prim, rays, any=any_hit, records=True, nthreads=8)
        recs = want["records"]
        w = f"{where} any={any_hit}"
        assert_hits_exact(gpu_trace(scene, rays, any_hit, True), want["hits"], w + " reflayout", recs)
        for c in range(len(Scene.kernel_configs())):
            try:
                scene.set_kernel_config(c)
            except Exception:                                  # a staged configuration may not fit a deep tree
                continue
            h = scene.hit(d, any=any_hit)
            got = h.cpu().numpy().view(L.hit_dtype).reshape(-1)
            assert_hits_exact(got, want["hits"], f"{w} cfg={c}", recs)
            h16 = scene.hit(d, any=any_hit, hit16=True).cpu().numpy().view(L.hit16_dtype).reshape(-1)
            assert np.array_equal(h16.view(np.uint8), L.pack_hit16(got).view(np.uint8)), f"{w} cfg={c} hit16"
            if c == 0:
                assert torch.equal(scene.hit(d, any=any_hit, sort=True).view(torch.int32), h.view(torch.int32)), w + " sort"
                cnt = torch.tensor([n], dtype=torch.int64, device="cuda:0")
                assert torch.equal(scene.hit_indirect(d, cnt, any=any_hit).view(torch.int32), h.view(torch.int32)), w + " indirect"
                if not any_hit:
                    assert_records_exact(scene, rays, h, want, w)
        scene.set_kernel_config(-1)
        os.environ["TRQ_CHUNK_RAYS"] = "4096"
        try:
            host = scene.hit(rays, any=any_hit)
        finally:
            del os.environ["TRQ_CHUNK_RAYS"]
        assert np.array_equal(host.view(np.uint8), hits_to_numpy(scene.hit(d, any=any_hit)).view(np.uint8)), w + " host path"
    scene.close()


# ------------------------------------------------------------------------------------------------------------- tests
def test_special_rays_every_path(built, port, capsys):
    _torch()
    rng = np.random.default_rng(2026)
    for name, prim, n, n_nan in _trace_scenes(rng):
        rays, fam = special_rays(rng, prim, n, n_nan_origin=n_nan if name != "comb31" else 0)
        if name == "comb31":
            rays = np.concatenate([rays, nan_origin_rays(rng, n_nan)])
        _check_all_paths(port, prim, rays, name)
    with capsys.disabled():
        print(f"\nsphere uv: largest error of phi (atan2f) seen {_seen['u']} ulp, of theta (asinf) {_seen['v']} ulp")


def test_poles_seams_and_flat_cubes(built, port, capsys):
    """Sphere hits on the poles (gn.y = +-1 and |gn.y| > 1) and on the seam (gn.x, gn.z at +-0), reached by rays along y
    with signed-zero components; cubes flat at -0.0 / +0.0 hit at t = 0 from their plane (the zero fminf / fmaxf pick in
    the local box test reaches uv)."""
    _torch()
    for name, (prim, rays) in (("poles", pole_spheres_scene()), ("flat cubes", flat_cube_scene())):
        _check_all_paths(port, prim, rays, name)
    with capsys.disabled():
        print(f"\nsphere uv: largest error of phi (atan2f) seen {_seen['u']} ulp, of theta (asinf) {_seen['v']} ulp")


def test_automatic_ordering_of_special_rays(built, port):
    """TRQ_AUTO_SORT=1 on 2^20 + 1 special rays: the ordered trace equals sort=False byte for byte, and the oracle on a
    subsample."""
    torch = _torch()
    from tracer_b200 import Scene, harness as H, rays_to_torch
    prim = H.scene_soup(20000, seed=8, extent=0.05)
    scene = Scene(prim, 0)
    rays, _ = special_rays(np.random.default_rng(5), prim, (1 << 20) + 1, n_nan_origin=64)
    d = rays_to_torch(rays, "cuda:0")
    os.environ["TRQ_AUTO_SORT"] = "1"
    try:
        for any_hit in (False, True):
            plain = scene.hit(d, any=any_hit, sort=False).clone()
            assert torch.equal(scene.hit(d, any=any_hit).view(torch.int32), plain.view(torch.int32)), any_hit
            assert torch.equal(scene.hit(d, any=any_hit, sort=True).view(torch.int32), plain.view(torch.int32)), any_hit
            sub = np.unique(np.concatenate([np.arange(0, rays.size, 61), np.nonzero(np.isnan(rays["o"]).any(axis=1))[0]]))
            want = port.trace(prim, np.ascontiguousarray(rays[sub]), any=any_hit, nthreads=8)["hits"]
            assert_hits_exact(plain.cpu().numpy().view(L.hit_dtype).reshape(-1)[sub], want, f"auto ordering any={any_hit}")
    finally:
        del os.environ["TRQ_AUTO_SORT"]
    scene.close()


def _spawned(out, src, cnt):
    n = int(cnt.item())
    s = src.cpu().numpy()[:n].astype(np.uint32)
    order = np.argsort(s, kind="stable")
    return out.cpu().numpy().view(L.ray_dtype).reshape(-1)[:n][order], s[order]


def _check_spawns(scene, prim, d, h, recs, light_a, light_b, where):
    """Spawn origins, shadow directions and lengths bit for bit against the host restatement on the device's own records,
    NaN-aware (a NaN that float arithmetic makes has no agreed payload: 0x7fffffff on the device, the input's on x86);
    bounce directions by the exact candidate test."""
    from tracer_b200 import harness as H
    for seed in (3, 1 << 20):
        got, src = _spawned(*scene.spawn_bounce(d, h, seed_base=seed))
        want, wsrc = H.bounce_rays(recs, seed_base=seed)
        assert np.array_equal(src, wsrc), where
        assert _nan_aware_equal(got["o"], want["o"]), f"{where}: bounce origins (offset_ray)"
        assert (got["tmax"] == f32(L.FLT_MAX)).all()
        assert_bounce_directions(got["d"], recs["sn"][src], src, seed, where)
        got, src = _spawned(*scene.spawn_shadow(d, h, light_a, light_b, seed_base=seed))
        want, wsrc = H.shadow_rays(recs, prim.squareList[light_a:light_a + 1], prim.squareList[light_b:light_b + 1], seed_base=seed)
        assert np.array_equal(src, wsrc), where
        assert _nan_aware_equal(got["o"], want["o"]), f"{where}: shadow origins (offset_ray)"
        assert _nan_aware_equal(got["d"], want["d"]), f"{where}: shadow directions"
        assert _nan_aware_equal(got["tmax"], want["tmax"]), f"{where}: shadow lengths"


def test_degenerate_surfaces_spawn_like_the_host(built, port):
    """Hits on triangles with NaN / zero / negative / huge vertex normals, spheres of radius 0, -1 and 1e-12 far from the
    origin, and cubes with a zero-scale or NaN matrix: records against the oracle, spawns against the host restatement."""
    _torch()
    from tracer_b200 import Scene, hits_to_numpy, rays_to_torch
    prim, targets = degenerate_scene()
    rays = aimed_rays(np.random.default_rng(2), targets, 6000)
    scene = Scene(prim, 0)
    d = rays_to_torch(rays, "cuda:0")
    h = scene.hit(d)
    want = port.trace(prim, rays, records=True, nthreads=8)
    assert_hits_exact(hits_to_numpy(h), want["hits"], "degenerate", want["records"])
    recs = assert_records_exact(scene, rays, h, want, "degenerate")
    _check_spawns(scene, prim, d, h, recs, 0, 1, "degenerate")
    scene.close()


def test_cornell_bounce_directions_exact(built):
    """The reference Cornell mix's primary hits: bounce directions by the exact candidate test (it replaces a 2e-3 bound)."""
    _torch()
    from tracer_b200 import Scene, harness as H
    prim = H.scene_reference_cornell()
    scene = Scene(prim, 0)
    d = scene.cast_rays((278, 278, -800), (278, 278, 278), (0, 1, 0), np.float32(45 * (np.pi / 180)), 320, 180)
    h = scene.hit(d)
    recs = scene.expand(d, h).cpu().numpy().view(L.record_dtype).reshape(-1)
    _check_spawns(scene, prim, d, h, recs, 5, 6, "cornell")
    scene.close()


def test_count_clamps(built):
    """trq_trace_indirect writes exactly min(*count, capacity) records and nothing beyond; the spawns clamp *d_n to n."""
    torch = _torch()
    from tracer_b200 import Scene, harness as H, rays_to_torch
    prim = H.scene_reference_cornell()
    scene = Scene(prim, 0)
    rays, _ = special_rays(np.random.default_rng(9), prim, 1000, n_nan_origin=8)
    d = rays_to_torch(rays, "cuda:0")
    cap = rays.size
    for any_hit in (False, True):
        full = scene.hit(d, any=any_hit)
        for count in (cap + 1, cap + 12345, cap, cap - 1, 1):
            out = torch.full((cap + 64, 8), 7.0, device="cuda:0")
            cnt = torch.tensor([count], dtype=torch.int64, device="cuda:0")
            scene.hit_indirect(d, cnt, any=any_hit, out=out)
            k = min(count, cap)
            assert torch.equal(out[:k].view(torch.int32), full[:k].view(torch.int32)), (count, any_hit)
            assert bool((out[k:] == 7.0).all()), (count, any_hit)
    h = scene.hit(d)
    hit = (h[:, 7].view(torch.int32) & 1).cpu().numpy()
    for fn, extra in ((scene.spawn_bounce, ()), (scene.spawn_shadow, (5, 6))):
        base = _spawned(*fn(d, h, *extra, seed_base=4))
        for over in (1, 1000, 1 << 40):
            cin = torch.tensor([cap + over], dtype=torch.int64, device="cuda:0")
            out = torch.full((cap + 64, 8), 7.0, device="cuda:0")
            got = _spawned(*fn(d, h, *extra, seed_base=4, count_in=cin, out=out))
            assert got[0].size == int(hit.sum()) == base[0].size
            assert np.array_equal(got[0].view(np.uint8), base[0].view(np.uint8)) and np.array_equal(got[1], base[1])
            assert bool((out[cap:] == 7.0).all())
    scene.close()
