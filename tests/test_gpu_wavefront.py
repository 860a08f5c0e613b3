"""GPU: the device ray producers at the wavefront workloads' sizes, for any camera, over several frames, on every scene
kind; and the wavefront wrappers' argument checks.

Rays and RNG texture bytes are compared with the host restatements (tracer_b200/harness.py) byte for byte, NaN-aware, on the
device's own records (trq_expand_hits); bounce directions by assert_bounce_directions where the device's bits differ from the
host's; hits by assert_hits_exact against port.trace(..., records=True). Spawned rays are ordered by srcIndex first. At full
size (c2: 1920x1080, c3path: 3840x2160 on scene_c3(2)) every produced ray is checked, and the hits of each wave on a subsample:
every 16th ray plus every sphere / cube / square hit. Rules and case families: tests/test_wavefront_cpu.py."""
import ctypes as C
import os

import numpy as np
import pytest

from tracer_b200 import layout as L

from .test_gpu_parity import _torch
from .test_gpu_special_rays import assert_bounce_directions, assert_hits_exact
from .test_special_rays_cpu import _nan_aware_equal
from .test_wavefront_cpu import (BENCH_CASTS, CAST_SIZES, CORNELL_CAMERA, C1_CAMERA, SEED_BASES, assert_rays_equal,
                                 assert_shadow_lengths, degenerate_cameras, host_camera_rays, pcg32_first_two, random_cameras,
                                 subsample)
from .util import bits

pytestmark = pytest.mark.gpu
f32 = np.float32
NTHREADS = max(8, os.cpu_count() or 8)


def _rays(t, n=None):
    a = t.detach().cpu().numpy().view(L.ray_dtype).reshape(-1)
    return np.ascontiguousarray(a if n is None else a[:n])


def _hits(t, n=None):
    a = t.detach().cpu().numpy().view(L.hit_dtype).reshape(-1)
    return np.ascontiguousarray(a if n is None else a[:n])


def _records(scene, rays, hits, n):
    """The device's own HitRecords of the first n rays (trq_expand_hits)."""
    return scene.expand(rays[:n], hits[:n]).cpu().numpy().view(L.record_dtype).reshape(-1)


def _spawned(out, src, cnt):
    n = int(cnt.item())
    s = src[:n].cpu().numpy().astype(np.uint32)
    order = np.argsort(s, kind="stable")
    return _rays(out, n)[order], s[order]


def _uu(seed_base, src):
    """The two draws of each ray, PCG32((seed_base + src) mod 2^64, 1)."""
    return pcg32_first_two((np.uint64(seed_base) + src.astype(np.uint64)) if src.size else np.zeros(0, np.uint64))


def check_bounce(got, src, want, wsrc, sn, where, seed_base=None, uu=None):
    """Bounce rays against the host restatement: srcIndex equal, origins and tmax bit for bit, directions equal to the
    host's or, where cosf / sinf gave other bits, one of the exact candidates."""
    assert np.array_equal(src, wsrc), f"{where}: srcIndex"
    assert _nan_aware_equal(got["o"].reshape(-1), want["o"].reshape(-1)), f"{where}: bounce origins"
    assert (got["tmax"] == f32(L.FLT_MAX)).all(), f"{where}: bounce tmax"
    other = np.nonzero(~(bits(got["d"]) == bits(want["d"])).all(axis=1))[0]
    for k in range(0, other.size, 1 << 17):                    # the candidate arrays are large: in pieces
        o = other[k:k + (1 << 17)]
        assert_bounce_directions(got["d"][o], sn[o], src[o], 0, where, uu=_uu(seed_base, src[o]) if uu is None else uu[o])


def check_shadow(got, src, want, wsrc, where):
    assert np.array_equal(src, wsrc), f"{where}: srcIndex"
    assert_rays_equal(got, want, where)
    assert_shadow_lengths(got["tmax"], want["tmax"], where)


def check_hits(port, prim, rays, got, any_hit, where, sub=None):
    if sub is not None:
        rays, got = np.ascontiguousarray(rays[sub]), got[sub]
    want = port.trace(prim, rays, any=any_hit, records=True, nthreads=NTHREADS)
    assert_hits_exact(got, want["hits"], where, want["records"])


# ------------------------------------------------------------------------------------------------------------ cameras
@pytest.fixture(scope="module")
def cornell(built):
    _torch()
    from tracer_b200 import Scene, harness as H
    prim = H.scene_reference_cornell()
    scene = Scene(prim, 0)
    yield prim, scene
    scene.close()


def _cast(scene, cam, W, H, **kw):
    frm, at, up, vfov, focus = cam
    return scene.cast_rays(frm, at, up, vfov, W, H, focus_dist=focus, **kw)


def test_camera_rays_for_any_camera(cornell):
    torch = _torch()
    prim, scene = cornell
    cases = [(f"random {k}", cam, W, H) for k, (cam, W, H) in enumerate(random_cameras(np.random.default_rng(11)))]
    cases += list(BENCH_CASTS)
    cases += [(f"{W}x{H}", CORNELL_CAMERA, W, H) for W, H in CAST_SIZES] + [(f"c1 {W}x{H}", C1_CAMERA, W, H) for W, H in CAST_SIZES]
    cases += [(f"degenerate: {f}", cam, W, H) for f, cam in degenerate_cameras() for W, H in ((33, 17), (4097, 3))]
    for where, cam, W, H in cases:
        assert_rays_equal(_rays(_cast(scene, cam, W, H)), host_camera_rays(cam, W, H), where)
    # a cast on a side stream equals one on the default stream
    side = torch.cuda.Stream()
    a = _cast(scene, CORNELL_CAMERA, 1920, 1080)
    out = torch.full((1920 * 1080, 8), 7.0, device="cuda:0")
    side.wait_stream(torch.cuda.current_stream())              # the sentinel fill before the cast
    _cast(scene, CORNELL_CAMERA, 1920, 1080, out=out, stream=side.cuda_stream)
    side.synchronize()
    assert torch.equal(out.view(torch.int32), a.view(torch.int32))


def test_camera_refusals_and_empty_images(cornell):
    torch = _torch()
    from tracer_b200._lib import ERR_INVALID, TrqError
    prim, scene = cornell
    out = torch.full((64, 8), 7.0, device="cuda:0")
    for aperture in (0.1, -1.0, float("nan")):
        with pytest.raises(TrqError) as e:
            _cast(scene, CORNELL_CAMERA, 8, 8, out=out, aperture=aperture)
        assert e.value.status == ERR_INVALID
    for W, H in ((0, 5), (5, 0), (0, 0)):
        _cast(scene, CORNELL_CAMERA, W, H, out=out)
    torch.cuda.synchronize()
    assert bool((out == 7.0).all()), "a refused or empty cast wrote rays"


# ------------------------------------------------------------------------------------------------ the bench's wavefronts
def _bench_step(scene, W, Hh, seed_base, bufs):
    """bench.py's Work.step for the device-resident workloads (c2, c3path), restated."""
    r0, h0, r1, h1, s1, c1 = bufs
    frm, at, up, vfov, _ = CORNELL_CAMERA
    scene.cast_rays(frm, at, up, vfov, W, Hh, out=r0)
    scene.hit(r0, out=h0)
    scene.spawn_bounce(r0, h0, seed_base=seed_base, out=r1, src=s1, count=c1)
    scene.hit_indirect(r1, c1, out=h1)


@pytest.mark.parametrize("workload", ["c2", "c3path"])
def test_bench_wavefront_at_full_size(built, port, workload, capsys):
    import time
    torch = _torch()
    from tracer_b200 import Scene, harness as H
    t_start = time.time()
    prim = H.scene_c2() if workload == "c2" else H.scene_c3(2)
    W, Hh = (1920, 1080) if workload == "c2" else (3840, 2160)
    scene = Scene(prim, 0)
    dev = "cuda:0"
    r0 = torch.empty((W * Hh, 8), dtype=torch.float32, device=dev); h0 = torch.empty_like(r0)
    r1 = torch.empty_like(r0); h1 = torch.empty_like(r0)
    s1 = torch.empty(W * Hh, dtype=torch.int32, device=dev); c1 = torch.zeros(1, dtype=torch.int64, device=dev)
    bufs = (r0, h0, r1, h1, s1, c1)
    primary = host_camera_rays(CORNELL_CAMERA, W, Hh)
    first = None
    for seed_base in SEED_BASES:
        where = f"{workload} seed_base={seed_base:#x}"
        _bench_step(scene, W, Hh, seed_base, bufs)
        torch.cuda.synchronize()
        if first is None:                                      # the primary wave does not depend on the seed: checked once
            assert_rays_equal(_rays(r0), primary, where + " camera")
            g0 = _hits(h0)
            check_hits(port, prim, primary, g0, False, where + " primary", subsample(W * Hh, g0["pType"]))
            recs0 = _records(scene, r0, h0, W * Hh)
            first = (r0.clone(), h0.clone())
        else:
            assert torch.equal(r0.view(torch.int32), first[0].view(torch.int32)) and torch.equal(h0.view(torch.int32), first[1].view(torch.int32))
        n1 = int(c1.item())
        want, wsrc = H.bounce_rays(recs0, seed_base=seed_base)
        assert n1 == want.size == int((recs0["hit"] == 1).sum()), where
        got, src = _spawned(r1, s1, c1)
        check_bounce(got, src, want, wsrc, recs0["sn"][wsrc], where + " bounce", seed_base=seed_base)
        g1 = _hits(h1, n1)
        check_hits(port, prim, _rays(r1, n1), g1, False, where + " bounce hits", subsample(n1, g1["pType"]))
        if seed_base == SEED_BASES[0]:                         # the step again on the same tensors: same count, same rays
            before = (got.copy(), src.copy())
            _bench_step(scene, W, Hh, seed_base, bufs)
            torch.cuda.synchronize()
            assert int(c1.item()) == n1
            again, asrc = _spawned(r1, s1, c1)
            assert np.array_equal(asrc, before[1]) and np.array_equal(again.view(np.uint8), before[0].view(np.uint8)), where + " repeated step"
    scene.close()
    with capsys.disabled():
        print(f"\n{workload}: {W}x{Hh}, {len(SEED_BASES)} seed bases, {time.time() - t_start:.0f} s")


# ------------------------------------------------------------------------------------------------------ every scene kind
def _wavefront(port, scene, prim, r0, seed, where, lights=None, hit16_wave=1):
    """r0 -> trace -> bounce -> trace_indirect (-> shadow toward `lights` -> any-hit trace_indirect), every wave checked.
    The wave numbered hit16_wave (1 bounce, 2 shadow) is also traced into trq_hit16 records, which must pack its trq_hit."""
    torch = _torch()
    from tracer_b200 import harness as H
    n0 = r0.shape[0]
    h0 = scene.hit(r0)
    check_hits(port, prim, _rays(r0), _hits(h0), False, where + " primary")
    recs0 = _records(scene, r0, h0, n0)
    r1, s1, c1 = scene.spawn_bounce(r0, h0, seed_base=seed)
    h1 = scene.hit_indirect(r1, c1)
    n1 = int(c1.item())
    assert n1 > 0, where
    got, src = _spawned(r1, s1, c1)
    want, wsrc = H.bounce_rays(recs0, seed_base=seed)
    check_bounce(got, src, want, wsrc, recs0["sn"][wsrc], where + " bounce", seed_base=seed)
    check_hits(port, prim, _rays(r1, n1), _hits(h1, n1), False, where + " bounce hits")
    waves = [(r1, c1, h1, n1, False)]
    if lights is not None:
        la, lb = lights
        recs1 = _records(scene, r1, h1, n1)
        sh, s2, c2 = scene.spawn_shadow(r1, h1, la, lb, seed_base=seed + 1, count_in=c1)
        occ = scene.hit_indirect(sh, c2, any=True)
        n2 = int(c2.item())
        got, src = _spawned(sh, s2, c2)
        want, wsrc = H.shadow_rays(recs1, prim.squareList[la:la + 1], prim.squareList[lb:lb + 1], seed_base=seed + 1)
        assert n2 == want.size > 0, where
        check_shadow(got, src, want, wsrc, where + " shadow")
        check_hits(port, prim, _rays(sh, n2), _hits(occ, n2), True, where + " shadow hits")
        waves.append((sh, c2, occ, n2, True))
    rays, cnt, h, n, any_hit = waves[hit16_wave - 1]
    h16 = scene.hit_indirect(rays, cnt, any=any_hit, hit16=True)
    torch.cuda.synchronize()
    assert np.array_equal(h16[:n].cpu().numpy().view(np.uint8).reshape(-1), L.pack_hit16(_hits(h, n)).view(np.uint8)), where + " hit16"


def test_every_scene_kind(built, port, capsys):
    _torch()
    from tracer_b200 import Scene, harness as H, rays_to_torch
    from .test_special_rays_cpu import _seen
    # C1: bounce rays from spheres only
    prim = H.scene_c1()
    scene = Scene(prim, 0)
    _wavefront(port, scene, prim, _cast(scene, C1_CAMERA, 640, 360), 5, "c1")
    scene.close()
    # C4: primary -> bounce -> any-hit shadow rays toward its lights (square list without leaves)
    prim = H.scene_c4(2)
    scene = Scene(prim, 0)
    _seen["u"] = _seen["v"] = 0
    _wavefront(port, scene, prim, _cast(scene, CORNELL_CAMERA, 480, 270), 1 << 32, "c4", lights=(5, 6), hit16_wave=2)
    scene.close()
    with capsys.disabled():
        print(f"\nC4 wavefront, sphere uv: largest error of phi (atan2f) {_seen['u']} ulp, of theta (asinf) {_seen['v']} ulp")
    # the reference's Cornell mix
    prim = H.scene_reference_cornell()
    scene = Scene(prim, 0)
    _wavefront(port, scene, prim, _cast(scene, CORNELL_CAMERA, 320, 180), SEED_BASES[-1], "cornell mix", lights=(5, 6))
    scene.close()
    # the cube with a down-scaling model matrix (test_gpu_producers.test_cube_with_a_down_scaling_model_matrix), rays inside it
    model = H.translation4x4(0.5, -0.25, 2.0) @ H.rotation4x4(0.3, (0, 1, 0)) @ H.scale4x4(0.01, 0.02, 0.015)
    c = H.make_cube(model, 3)
    c["box_mini"], c["box_maxi"] = (-100, -60, -80), (100, 60, 80)
    prim = H.build_primitive(cubes=np.array([c, H.cornell_cubes()[0]], dtype=L.cube_dtype))
    rng = np.random.default_rng(5)
    n = 20000
    rays = np.zeros(n, dtype=L.ray_dtype)
    local = rng.uniform([-95, -55, -75], [95, 55, 75], size=(n, 3))
    M = model.astype(np.float64)
    rays["o"] = ((M[:3, :3] @ local.T).T + M[:3, 3]).astype(f32)
    d = rng.normal(size=(n, 3))
    rays["d"] = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(f32)
    rays["tmax"] = rng.uniform(0.5, 150.0, size=n).astype(f32)
    scene = Scene(prim, 0)
    _wavefront(port, scene, prim, rays_to_torch(rays, "cuda:0"), 3, "down-scaled cube")
    scene.close()


# ----------------------------------------------------------------------------------------------- RNG texture, 3 frames
def _texture_draws(texels):
    """The first two randomF of each texel's stream (exRNG layout: state hi, lo, inc hi, lo), PCG32 in Python integers."""
    out = np.zeros((len(texels), 2), dtype=f32)
    for k, t in enumerate(texels.astype(np.uint64)):
        state, inc = (int(t[0]) << 32) | int(t[1]), (int(t[2]) << 32) | int(t[3])
        for j in range(2):
            old = state
            state = (old * 6364136223846793005 + inc) & 0xFFFFFFFFFFFFFFFF
            x = (((old >> 18) ^ old) >> 27) & 0xFFFFFFFF
            rot = old >> 59
            r = ((x >> rot) | (x << ((-rot) & 31))) & 0xFFFFFFFF
            out[k, j] = f32(np.uint32(r)) * f32(2.0 ** -32)
    return out


def test_rng_state_texture_three_frames(cornell, port):
    """Three frames of rng_frame_begin -> primary -> bounce -> shadow -> second bounce -> shadow at 320x180, pixel_of chained
    through each wave's srcIndex: after every wave the texture equals the host's, and exactly the pixels that drew changed."""
    torch = _torch()
    from tracer_b200 import harness as H
    prim, scene = cornell
    W, Hh = 320, 180
    la, lb = 5, 6
    tex0 = np.random.default_rng(21).integers(0, 1 << 32, size=(W * Hh, 4), dtype=np.uint64).astype(np.uint32)
    tex_d = torch.from_numpy(tex0.view(np.int32)).to("cuda:0")
    tex_h = tex0.copy()
    twice = tex_d.clone()
    scene.rng_frame_begin(twice); scene.rng_frame_begin(twice)
    assert torch.equal(twice, tex_d), "rng_frame_begin twice is the identity"

    def texture_equal(where):
        assert np.array_equal(tex_d.cpu().numpy().view(np.uint32), tex_h), f"RNG texture after {where}"

    def drew(before, pixels, where):
        changed = np.nonzero((tex_h != before).any(axis=1))[0]
        assert np.array_equal(changed, np.unique(pixels)), f"{where}: the pixels that drew, and only they, change"

    for frame in range(3):
        f = f"frame {frame}"
        scene.rng_frame_begin(tex_d); H.rng_frame_begin(tex_h)
        texture_equal(f + " begin")
        r0 = _cast(scene, CORNELL_CAMERA, W, Hh)
        h0 = scene.hit(r0)
        recs = _records(scene, r0, h0, W * Hh)
        rays, hits, cnt, pix, n = r0, h0, None, None, W * Hh     # pix: the pixel of each ray of the current wave (None: i)
        for depth in (1, 2):
            w = f"{f} bounce {depth}"
            before = tex_h.copy()
            r, s, c = scene.spawn_bounce(rays, hits, count_in=cnt, pixel_of=pix, rng_state=tex_d)
            want, wpix = H.bounce_rays(recs, pixel_of=None if pix is None else pix[:n].cpu().numpy().astype(np.uint32), rng_state=tex_h)
            texture_equal(w)
            drew(before, wpix, w)
            got, gpix = _spawned(r, s, c)
            order = np.argsort(wpix, kind="stable")
            ray_of_pixel = np.empty(W * Hh, dtype=np.int64)
            ray_of_pixel[np.arange(n) if pix is None else pix[:n].cpu().numpy()] = np.arange(n)
            check_bounce(got, gpix, want[order], wpix[order], recs["sn"][ray_of_pixel[gpix]], w, uu=_texture_draws(before[gpix]))
            n1 = int(c.item())
            h = scene.hit_indirect(r, c)
            check_hits(port, prim, _rays(r, n1), _hits(h, n1), False, w + " hits")
            recs1 = _records(scene, r, h, n1)
            w = f"{f} shadow {depth}"
            before = tex_h.copy()
            sh, s2, c2 = scene.spawn_shadow(r, h, la, lb, count_in=c, pixel_of=s, rng_state=tex_d)
            want, wpix = H.shadow_rays(recs1, prim.squareList[la:la + 1], prim.squareList[lb:lb + 1],
                                       pixel_of=s[:n1].cpu().numpy().astype(np.uint32), rng_state=tex_h)
            texture_equal(w)
            drew(before, wpix, w)
            got, gpix = _spawned(sh, s2, c2)
            order = np.argsort(wpix, kind="stable")
            check_shadow(got, gpix, want[order], wpix[order], w)
            occ = scene.hit_indirect(sh, c2, any=True)
            check_hits(port, prim, _rays(sh, int(c2.item())), _hits(occ, int(c2.item())), True, w + " hits")
            rays, hits, cnt, pix, n, recs = r, h, c, s, n1, recs1
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------------------------- wrapper arguments
def _sentinel(torch, shape, dtype):
    t = torch.empty(shape, dtype=dtype, device="cuda:0")
    t.view(torch.uint8).fill_(0xA5)
    return t


def test_wrapper_arguments_are_refused_before_any_launch(cornell):
    """Every refusal is a TypeError / ValueError raised before a launch. Each bad argument lies inside a larger sentinel
    buffer the test owns, so even an unchecked call would stay inside allocated memory; the sentinels must be intact."""
    torch = _torch()
    from tracer_b200 import launch_count
    prim, scene = cornell
    n = 1000
    rays = _cast(scene, CORNELL_CAMERA, 50, 20)
    hits = scene.hit(rays)
    torch.cuda.synchronize()
    big = _sentinel(torch, (2 * n, 8), torch.float32)               # rays / hits / out
    big16 = _sentinel(torch, (2 * n, 4), torch.float32)              # trq_hit16-shaped, with 32-byte rows of room behind it
    wide = _sentinel(torch, (n, 16), torch.float32)                  # non-contiguous (n, 8) views
    ints = _sentinel(torch, (2 * n,), torch.int32)                   # src / pixel_of
    longs = _sentinel(torch, (2 * n,), torch.int64)                  # an int32 view inside stays inside
    tex = _sentinel(torch, (2 * n, 8), torch.int32)                  # rng_state
    recs = _sentinel(torch, (2 * n, 16), torch.float32)
    dbl = _sentinel(torch, (n, 8), torch.float64)
    pixels = torch.arange(2 * n, dtype=torch.int32, device="cuda:0")   # valid pixels of `tex`
    count = torch.tensor([n], dtype=torch.int64, device="cuda:0")
    sentinels = [big, big16, wide, ints, longs, tex, recs, dbl, pixels]
    snap = [t.clone() for t in sentinels] + [rays.clone(), hits.clone(), count.clone()]
    cases = [
        ("hit out undersized", ValueError, lambda: scene.hit(rays, out=big[:n - 1])),
        ("hit out trq_hit16 width for trq_hit", TypeError, lambda: scene.hit(rays, out=big16[:n])),
        ("hit out float64", TypeError, lambda: scene.hit(rays, out=dbl)),
        ("hit out is rays", ValueError, lambda: scene.hit(big[:n], out=big[n // 2: n // 2 + n])),
        ("hit rays non-contiguous", TypeError, lambda: scene.hit(wide[:, :8])),
        ("indirect count int32", TypeError, lambda: scene.hit_indirect(rays, longs[:1].view(torch.int32)[:1], out=big[:n])),
        ("indirect count two elements", ValueError, lambda: scene.hit_indirect(rays, longs[:2], out=big[:n])),
        ("indirect out undersized", ValueError, lambda: scene.hit_indirect(rays, count, out=big[:n - 1])),
        ("indirect hit16 out of trq_hit width", TypeError, lambda: scene.hit_indirect(rays, count, out=big[:n], hit16=True)),
        ("indirect out overlaps rays", ValueError, lambda: scene.hit_indirect(big[:n], count, out=big[n - 1: 2 * n - 1])),
        ("spawn hits in trq_hit16", TypeError, lambda: scene.spawn_bounce(rays, big16[:n], out=big[:n], src=ints[:n], count=longs[:1])),
        ("spawn hits too few", ValueError, lambda: scene.spawn_bounce(rays, hits[:n - 1], out=big[:n], src=ints[:n], count=longs[:1])),
        ("spawn count int32", TypeError, lambda: scene.spawn_bounce(rays, hits, out=big[:n], src=ints[:n], count=longs[:1].view(torch.int32)[:1])),
        ("spawn count_in int32", TypeError, lambda: scene.spawn_bounce(rays, hits, count_in=longs[:1].view(torch.int32)[:1], out=big[:n], src=ints[:n], count=longs[1:2])),
        ("spawn count is count_in", ValueError, lambda: scene.spawn_bounce(rays, hits, count_in=longs[:1], out=big[:n], src=ints[:n], count=longs[:1])),
        ("spawn out undersized", ValueError, lambda: scene.spawn_bounce(rays, hits, out=big[:n - 1], src=ints[:n], count=longs[:1])),
        ("spawn out is rays", ValueError, lambda: scene.spawn_bounce(big[:n], hits, out=big[:n], src=ints[:n], count=longs[:1])),
        ("spawn out overlaps hits", ValueError, lambda: scene.spawn_shadow(rays, big[:n], 5, 6, out=big[n - 1:2 * n - 1], src=ints[:n], count=longs[:1])),
        ("spawn src int64", TypeError, lambda: scene.spawn_bounce(rays, hits, out=big[:n], src=longs[:n], count=longs[n:n + 1])),
        ("spawn src too short", ValueError, lambda: scene.spawn_bounce(rays, hits, out=big[:n], src=ints[:n - 1], count=longs[:1])),
        ("spawn src overlaps out", ValueError, lambda: scene.spawn_bounce(rays, hits, out=big[:n], src=big[:n].view(torch.int32).reshape(-1)[:n], count=longs[:1])),
        ("spawn pixel_of too short", ValueError, lambda: scene.spawn_bounce(rays, hits, pixel_of=pixels[:n - 1], rng_state=tex.view(-1)[:8 * n].view(2 * n, 4), out=big[:n], src=ints[:n], count=longs[:1])),
        ("spawn pixel_of int64", TypeError, lambda: scene.spawn_bounce(rays, hits, pixel_of=longs[:n], out=big[:n], src=ints[:n], count=longs[n:n + 1])),
        ("spawn pixel_of is src", ValueError, lambda: scene.spawn_bounce(rays, hits, pixel_of=ints[:n], out=big[:n], src=ints[:n], count=longs[:1])),
        ("spawn rng_state flat", TypeError, lambda: scene.spawn_bounce(rays, hits, rng_state=tex.view(-1)[:4 * n], out=big[:n], src=ints[:n], count=longs[:1])),
        ("spawn rng_state non-contiguous", TypeError, lambda: scene.spawn_bounce(rays, hits, rng_state=tex[:n, :4], out=big[:n], src=ints[:n], count=longs[:1])),
        ("spawn rng_state int64", TypeError, lambda: scene.spawn_bounce(rays, hits, rng_state=tex[:n].view(torch.int64), out=big[:n], src=ints[:n], count=longs[:1])),
        ("spawn rng_state too few pixels", ValueError, lambda: scene.spawn_bounce(rays, hits, rng_state=tex.view(-1)[:4 * (n - 1)].view(n - 1, 4), out=big[:n], src=ints[:n], count=longs[:1])),
        ("rng_frame_begin int64", TypeError, lambda: scene.rng_frame_begin(tex[:n].view(torch.int64))),
        ("rng_frame_begin flat", TypeError, lambda: scene.rng_frame_begin(tex.view(-1)[:4 * n])),   # unchecked: 4n texels of 16 B
        ("expand hits in trq_hit16", TypeError, lambda: scene.expand(rays, big16[:n], out=recs[:n])),
        ("expand out undersized", ValueError, lambda: scene.expand(rays, hits, out=recs[:n - 1])),
        ("cast out undersized", ValueError, lambda: scene.cast_rays((0, 0, -5), (0, 0, 0), (0, 1, 0), 0.5, 50, 20, out=big[:n - 1])),
        ("cast out float64", TypeError, lambda: scene.cast_rays((0, 0, -5), (0, 0, 0), (0, 1, 0), 0.5, 10, 10, out=longs[:800].view(torch.float64).view(100, 8))),
        ("update_vertices from pinned host memory", TypeError, lambda: scene.update_vertices(torch.from_numpy(prim.triList.view(np.uint8).reshape(-1).copy()).pin_memory())),
        ("rebuild from pinned host memory", TypeError, lambda: scene.rebuild(torch.from_numpy(prim.triList.view(np.uint8).reshape(-1).copy()).pin_memory())),
        ("update_vertices partial records", TypeError, lambda: scene.update_vertices(big.view(torch.uint8).reshape(-1)[:33])),
    ]
    for where, exc, call in cases:
        before = launch_count()
        with pytest.raises(exc):
            call()
        assert launch_count() == before, f"{where}: launched"
        torch.cuda.synchronize()
        for t, s in zip(sentinels + [rays, hits, count], snap):
            assert torch.equal(t.view(torch.uint8), s.view(torch.uint8)), f"{where}: a sentinel changed"
    # the checks pass what they should: the same buffers, well formed
    scene.spawn_bounce(rays, hits, out=big[:n], src=ints[:n], count=longs[:1])
    scene.hit_indirect(big[:n], longs[:1], out=big[n:])
    torch.cuda.synchronize()
    assert 0 < int(longs[0].item()) <= n


def test_shared_counter_spawns_nothing(cornell):
    """At the C-ABI, d_n == d_count: the spawn zeroes the counter on the stream before its kernel reads it, so it spawns
    nothing and writes nothing to out (include/tracer_rq.h)."""
    torch = _torch()
    from tracer_b200._lib import check, lib
    prim, scene = cornell
    rays = _cast(scene, CORNELL_CAMERA, 64, 32)
    hits = scene.hit(rays)
    n = rays.shape[0]
    for fn, extra in ((lib.trq_spawn_bounce, ()), (lib.trq_spawn_shadow, (5, 6))):
        out = _sentinel(torch, (n, 8), torch.float32)
        src = _sentinel(torch, (n,), torch.int32)
        keep = (out.clone(), src.clone())
        cnt = torch.tensor([n], dtype=torch.int64, device="cuda:0")
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        check(fn(scene._h, rays.data_ptr(), hits.data_ptr(), n, cnt.data_ptr(), 3, *extra, out.data_ptr(), src.data_ptr(),
                 cnt.data_ptr(), stream), fn.__name__)
        torch.cuda.synchronize()
        assert int(cnt.item()) == 0, fn.__name__
        assert torch.equal(out.view(torch.int32), keep[0].view(torch.int32)) and torch.equal(src, keep[1]), fn.__name__
