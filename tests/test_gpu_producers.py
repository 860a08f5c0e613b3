"""GPU: device-side ray producers (row f-3: castRay, bounce spawn, shadow spawn) and the device-resident wavefront
(trq_trace_indirect), against the host restatements in csrc/host/harness.cpp -- which tests/test_harness.py checks
against the reference's own functions -- and against the oracle for the traversal of the produced rays."""
import numpy as np
import pytest

from tracer_b200 import layout as L

from .test_gpu_special_rays import assert_bounce_directions
from .util import bits

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.fixture(scope="module")
def cornell(built):
    _torch()
    from tracer_b200 import Scene, harness as H
    prim = H.scene_reference_cornell()
    return prim, Scene(prim, 0)


def _np_rays(t, n=None):
    a = t.detach().cpu().numpy().view(L.ray_dtype).reshape(-1)
    return a if n is None else a[:n]


def test_cast_rays_bit_exact(cornell):
    from tracer_b200 import harness as H
    prim, scene = cornell
    dev = scene.cast_rays((278, 278, -800), (278, 278, 278), (0, 1, 0), np.float32(45 * (np.pi / 180)), 320, 180)
    host = H.cornell_camera_rays(320, 180)
    assert np.array_equal(_np_rays(dev).view(np.uint8), host.view(np.uint8))


def test_spawn_bounce_and_shadow_match_host(cornell):
    torch = _torch()
    from tracer_b200 import harness as H
    prim, scene = cornell
    d = scene.cast_rays((278, 278, -800), (278, 278, 278), (0, 1, 0), np.float32(45 * (np.pi / 180)), 320, 180)
    hits = scene.hit(d)
    recs = scene.expand(d, hits).cpu().numpy().view(L.record_dtype).reshape(-1)
    for kind in ("bounce", "shadow"):
        if kind == "bounce":
            out, src, cnt = scene.spawn_bounce(d, hits, seed_base=11)
            want, wsrc = H.bounce_rays(recs, seed_base=11)
        else:
            out, src, cnt = scene.spawn_shadow(d, hits, 5, 6, seed_base=11)
            want, wsrc = H.shadow_rays(recs, prim.squareList[5:6], prim.squareList[6:7], seed_base=11)
        n = int(cnt.item())
        assert n == want.size == int(recs["hit"].sum())
        got = _np_rays(out, n)
        order = np.argsort(src.cpu().numpy()[:n].astype(np.uint32), kind="stable")      # compaction order is warp-arrival order
        got = got[order]
        assert np.array_equal(src.cpu().numpy()[:n].astype(np.uint32)[order], wsrc)
        assert np.array_equal(bits(got["o"]), bits(want["o"])), "offset_ray origins must be bit-exact"
        if kind == "shadow":
            assert np.array_equal(bits(got["tmax"]), bits(want["tmax"])), "shadow lengths: strict fp32 sqrtf, bit-exact"
            assert np.array_equal(bits(got["d"]), bits(want["d"])), "shadow directions use no libm: bit-exact"
        else:
            assert (got["tmax"] == np.float32(L.FLT_MAX)).all()
            # cosf / sinf differ from libm by ulps: the direction must be one of the float32 chain's outcomes for cosf / sinf
            # within their documented error of cos / sin
            assert_bounce_directions(got["d"], recs["sn"][wsrc], wsrc, 11, "bounce")


def test_device_wavefront_two_bounces(cornell, port):
    """cast -> trace -> spawn -> trace_indirect -> spawn(indirect) -> trace_indirect with no host sync in between;
    every wave is checked bit-exactly against the oracle on the rays the device produced."""
    torch = _torch()
    from tracer_b200 import hits_to_numpy
    prim, scene = cornell
    W, H = 256, 144
    r0 = scene.cast_rays((278, 278, -800), (278, 278, 278), (0, 1, 0), np.float32(45 * (np.pi / 180)), W, H)
    h0 = scene.hit(r0)
    r1, s1, c1 = scene.spawn_bounce(r0, h0, seed_base=1)
    h1 = scene.hit_indirect(r1, c1)
    r2, s2, c2 = scene.spawn_bounce(r1, h1, seed_base=1 << 20, count_in=c1)
    h2 = scene.hit_indirect(r2, c2)
    sh, s3, c3 = scene.spawn_shadow(r1, h1, 5, 6, seed_base=7, count_in=c1)
    occ = scene.hit_indirect(sh, c3, any=True)
    torch.cuda.synchronize()
    n1, n2, n3 = int(c1.item()), int(c2.item()), int(c3.item())
    assert 0 < n2 < n1 < W * H and n3 == n2                      # every first-bounce hit spawns one bounce and one shadow ray
    for rays_t, hits_t, n, any_hit in ((r0, h0, W * H, False), (r1, h1, n1, False), (r2, h2, n2, False), (sh, occ, n3, True)):
        rays = _np_rays(rays_t, n).copy()
        got = hits_to_numpy(hits_t)[:n]
        want = port.trace(prim, rays, any=any_hit, nthreads=8)["hits"]
        for k in ("flags", "pType", "pIndex", "leafNode", "material"):
            assert np.array_equal(got[k], want[k]), k
        assert np.array_equal(bits(got["t"]), bits(want["t"]))
    # an indirect count of zero traces nothing and touches nothing
    zero = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    sentinel = torch.full((64, 8), 7.0, device="cuda:0")
    scene.hit_indirect(r1[:64].contiguous(), zero, out=sentinel)
    torch.cuda.synchronize()
    assert bool((sentinel == 7.0).all())


def _texture_draws(texels):
    """The first two randomF of each texel's stream (exRNG layout: state hi, lo, inc hi, lo), PCG32 in Python integers."""
    out = np.zeros((len(texels), 2), dtype=np.float32)
    for k, t in enumerate(texels.astype(np.uint64)):
        state, inc = (int(t[0]) << 32) | int(t[1]), (int(t[2]) << 32) | int(t[3])
        for j in range(2):
            old = state
            state = (old * 6364136223846793005 + inc) & 0xFFFFFFFFFFFFFFFF
            x = (((old >> 18) ^ old) >> 27) & 0xFFFFFFFF
            rot = old >> 59
            r = ((x >> rot) | (x << ((-rot) & 31))) & 0xFFFFFFFF
            out[k, j] = np.float32(np.uint32(r)) * np.float32(2.0 ** -32)
    return out


def test_rng_state_texture_two_waves(cornell):
    """Row f-4: the device spawns draw from and advance the reference's per-pixel RNG texture (Render.hh:96-120),
    wave after wave, exactly like the host restatement: state bytes identical, same rays, srcIndex = pixel."""
    torch = _torch()
    from tracer_b200 import harness as H
    prim, scene = cornell
    W, Hh = 320, 180
    d = scene.cast_rays((278, 278, -800), (278, 278, 278), (0, 1, 0), np.float32(45 * (np.pi / 180)), W, Hh)
    hits = scene.hit(d)
    rng = np.random.default_rng(9)
    tex0 = rng.integers(0, 1 << 32, size=(W * Hh, 4), dtype=np.uint64).astype(np.uint32)
    tex_d = torch.from_numpy(tex0.view(np.int32)).to("cuda:0")
    tex_h = tex0.copy()
    scene.rng_frame_begin(tex_d); H.rng_frame_begin(tex_h)             # the reference's kernel-entry conversion, once per frame
    assert np.array_equal(tex_d.cpu().numpy().view(np.uint32), tex_h) and np.array_equal(tex_h[:, :2], tex0[:, 2:])
    begun = tex_h.copy()
    # wave 1: bounce rays of the primary hits
    r1, s1, c1 = scene.spawn_bounce(d, hits, rng_state=tex_d)
    recs0 = scene.expand(d, hits).cpu().numpy().view(L.record_dtype).reshape(-1)
    w1, ws1 = H.bounce_rays(recs0, rng_state=tex_h)
    n1 = int(c1.item())
    assert n1 == w1.size
    assert np.array_equal(tex_d.cpu().numpy().view(np.uint32), tex_h), "RNG texture after wave 1"
    src1 = s1.cpu().numpy()[:n1].astype(np.uint32)
    order = np.argsort(src1, kind="stable")
    assert np.array_equal(src1[order], ws1)
    g1 = _np_rays(r1, n1)[order]
    assert np.array_equal(bits(g1["o"]), bits(w1["o"]))
    assert_bounce_directions(g1["d"], recs0["sn"][ws1], ws1, 0, "wave 1", uu=_texture_draws(begun[ws1]))
    # wave 2: shadow rays of the bounce hits, routed to their pixels through pixel_of = srcIndex of wave 1
    h1 = scene.hit_indirect(r1, c1)
    sh, s2, c2 = scene.spawn_shadow(r1, h1, 5, 6, count_in=c1, pixel_of=s1, rng_state=tex_d)
    n2 = int(c2.item())
    r1_np = _np_rays(r1, n1).copy()
    recs1 = scene.expand(r1_np, np.ascontiguousarray(h1.cpu().numpy().view(L.hit_dtype).reshape(-1)[:n1]))
    w2, ws2 = H.shadow_rays(recs1, prim.squareList[5:6], prim.squareList[6:7], pixel_of=src1, rng_state=tex_h)
    assert n2 == w2.size and 0 < n2 < n1
    assert np.array_equal(tex_d.cpu().numpy().view(np.uint32), tex_h), "RNG texture after wave 2"
    src2 = s2.cpu().numpy()[:n2].astype(np.uint32)
    order2 = np.argsort(src2, kind="stable")
    assert np.array_equal(src2[order2], np.sort(ws2))                   # pixels, not ray indices
    g2 = _np_rays(sh, n2)[order2]
    w2s = w2[np.argsort(ws2, kind="stable")]
    assert np.array_equal(bits(g2["o"]), bits(w2s["o"])) and np.array_equal(bits(g2["d"]), bits(w2s["d"]))
    assert (tex_h != begun).any(axis=1).sum() == n1                      # exactly the pixels that hit drew numbers


def test_device_wavefront_triangle_only_scene(built, port):
    """The same wavefront on a triangle-only scene (C2), where the trace kernel finishes its own records (no resolve
    pass): indirect batch sizes, closest and any-hit, against the oracle."""
    torch = _torch()
    from tracer_b200 import Scene, harness as H, hits_to_numpy
    prim = H.scene_c2()
    scene = Scene(prim, 0)
    assert scene.info["nTri"] == scene.info["nLeaf"]
    W, Hh = 320, 180
    r0 = scene.cast_rays((278, 278, -800), (278, 278, 278), (0, 1, 0), np.float32(45 * (np.pi / 180)), W, Hh)
    h0 = scene.hit(r0)
    r1, s1, c1 = scene.spawn_bounce(r0, h0, seed_base=5)
    h1 = scene.hit_indirect(r1, c1)
    a1 = scene.hit_indirect(r1, c1, any=True)
    s_h1 = scene.hit_indirect(r1, c1, sort=True)
    torch.cuda.synchronize()
    n1 = int(c1.item())
    assert 0 < n1 < W * Hh
    assert torch.equal(s_h1[:n1].view(torch.int32), h1[:n1].view(torch.int32))
    for rays_t, hits_t, n, any_hit in ((r0, h0, W * Hh, False), (r1, h1, n1, False), (r1, a1, n1, True)):
        rays = _np_rays(rays_t, n).copy()
        got = hits_to_numpy(hits_t)[:n]
        want = port.trace(prim, rays, any=any_hit, nthreads=8)["hits"]
        for k in ("flags", "pType", "pIndex", "leafNode", "material"):
            assert np.array_equal(got[k], want[k]), k
        for k in ("t", "u", "v"):
            assert np.array_equal(bits(got[k]), bits(want[k])), k
    scene.close()


def test_cube_with_a_down_scaling_model_matrix(built, port):
    """Cube::hit_test hands the CALLER's range.y to its local-space box test (Cube.hh:25, AABB.hh:116-145). When the model
    matrix scales down, a ray that starts inside the cube with range.y below the local exit distance is accepted at local
    t = range.y with axisPick = 0 -- an outcome that running the test again with another range.y does not reproduce (half of
    the hits below). trq_trace sees the real range; trq_expand_hits and the spawns rebuild those records from (t, u, v)
    (intersect.cuh: cube_surface). All three must give the oracle's records bit for bit."""
    torch = _torch()
    from tracer_b200 import Scene, harness as H, hits_to_numpy, rays_to_torch
    model = H.translation4x4(0.5, -0.25, 2.0) @ H.rotation4x4(0.3, (0, 1, 0)) @ H.scale4x4(0.01, 0.02, 0.015)
    c = H.make_cube(model, 3)
    c["box_mini"], c["box_maxi"] = (-100, -60, -80), (100, 60, 80)
    prim = H.build_primitive(cubes=np.array([c, H.cornell_cubes()[0]], dtype=L.cube_dtype))
    rng = np.random.default_rng(5)
    n = 20000
    rays = np.zeros(n, dtype=L.ray_dtype)
    local = rng.uniform([-95, -55, -75], [95, 55, 75], size=(n, 3))
    M = model.astype(np.float64)
    rays["o"] = ((M[:3, :3] @ local.T).T + M[:3, 3]).astype(np.float32)
    d = rng.normal(size=(n, 3))
    rays["d"] = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    rays["tmax"] = rng.uniform(0.5, 150.0, size=n).astype(np.float32)
    want = port.trace(prim, rays, records=True, nthreads=8)
    unclipped = rays.copy(); unclipped["tmax"] = L.FLT_MAX
    other = port.trace(prim, unclipped, records=True, nthreads=8)["records"]
    m = want["records"]["hit"] == 1
    clipped = m & ~np.all(bits(want["records"]["p"]) == bits(other["p"]), axis=1)
    assert clipped.sum() > n // 4, "the case under test must actually occur"

    scene = Scene(prim, 0)
    dr = rays_to_torch(rays, "cuda:0")
    dh = scene.hit(dr)
    hits = hits_to_numpy(dh)
    for k in want["hits"].dtype.names:
        assert np.array_equal(bits(hits[k]), bits(want["hits"][k])), k
    recs = scene.expand(dr, dh).cpu().numpy().view(L.record_dtype).reshape(-1)
    assert np.array_equal(recs["hit"], want["records"]["hit"])
    for k in ("t", "p", "gn", "sn", "uv", "front", "material"):
        assert np.array_equal(bits(recs[k][m]), bits(want["records"][k][m])), k
    out, src, cnt = scene.spawn_bounce(dr, dh, seed_base=3)
    wrays, wsrc = H.bounce_rays(want["records"], seed_base=3)
    k = int(cnt.item())
    assert k == wrays.size
    order = np.argsort(src.cpu().numpy()[:k].astype(np.uint32), kind="stable")
    got = _np_rays(out, k)[order]
    assert np.array_equal(src.cpu().numpy()[:k].astype(np.uint32)[order], wsrc)
    assert np.array_equal(bits(got["o"]), bits(wrays["o"]))
    scene.close()
