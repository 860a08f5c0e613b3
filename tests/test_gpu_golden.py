"""GPU: the CUDA path (through the C-ABI) against the golden vectors produced by the reference's own headers
(tests/golden/rq_golden.npz), and size-independent properties at BASELINE's full C3 size."""
import numpy as np
import pytest

from tracer_b200 import layout as L

from .util import CASES, assert_records_match_reference, bits, golden_case

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.mark.parametrize("reflayout", [False, True])
@pytest.mark.parametrize("name", CASES)
def test_gpu_matches_reference_golden(built, name, reflayout):
    torch = _torch()
    from tracer_b200 import Scene, hits_to_numpy, rays_to_torch
    prim, rays, any_hit, want = golden_case(name)
    scene = Scene(prim, 0)
    d = rays_to_torch(rays, "cuda:0")
    h = scene.hit(d, any=any_hit, reflayout=reflayout)
    hits = hits_to_numpy(h)
    hit = (hits["flags"] & 1) == 1
    assert np.array_equal(hit, want["hit"] == 1), "miss flags must be bit-exact"
    assert np.array_equal(bits(hits["t"][hit]), bits(want["t"][hit]))
    assert np.array_equal(hits["material"][hit], want["material"][hit])
    assert np.array_equal(((hits["flags"] >> 1) & 1)[hit], want["front"][hit])
    recs = scene.expand(d, h).cpu().numpy().view(L.record_dtype).reshape(-1)
    assert_records_match_reference(recs, want, hits=hits, where=name)
    scene.close()


@pytest.fixture(scope="module")
def c3(built):
    _torch()
    from tracer_b200 import Scene, harness as H, rays_to_torch
    prim = H.scene_c3(2)
    scene = Scene(prim, 0)
    primary = H.cornell_camera_rays(3840, 2160)
    d = rays_to_torch(primary, "cuda:0")
    recs = scene.expand(d, scene.hit(d)).cpu().numpy().view(L.record_dtype).reshape(-1)
    bounce, _ = H.bounce_rays(recs)
    return prim, scene, bounce


def test_c3_full_size_properties(c3, port):
    """BASELINE C3 at full size (1.0 M triangles, ~6.2 M incoherent bounce rays)."""
    torch = _torch()
    from tracer_b200 import hits_to_numpy, rays_to_torch
    prim, scene, rays = c3
    assert prim.nTri > 1_000_000 and rays.size > 6_000_000
    d = rays_to_torch(rays, "cuda:0")
    a = scene.hit(d)
    b = scene.hit(d)
    assert torch.equal(a, b), "not idempotent"
    r = scene.hit(d, reflayout=True)
    assert torch.equal(a, r), "packed kernel and reference-layout transcription disagree"
    anyh = scene.hit(d, any=True)
    ai, ci = anyh.view(torch.int32), a.view(torch.int32)
    assert torch.equal(ai[:, 7] & 1, ci[:, 7] & 1), "any-hit flag != closest-hit flag at tmax = FLT_MAX"
    hit = (ci[:, 7] & 1) == 1
    assert bool((anyh[hit, 0] >= a[hit, 0]).all()), "an any-hit t is closer than the closest hit"
    # sharding: tracing the two halves separately gives the same bytes as the whole batch
    half = rays.size // 2
    parts = torch.cat([scene.hit(d[:half].contiguous()), scene.hit(d[half:].contiguous())])
    assert torch.equal(parts, a)
    # host-pointer path (chunked, three streams) == device path
    host = scene.hit(rays)
    assert np.array_equal(host.view(np.uint8), hits_to_numpy(a).view(np.uint8))
    # oracle on a strided 1% sample: ids and t bit-exact
    sub = np.ascontiguousarray(rays[::97])
    want = port.trace(prim, sub, nthreads=8)["hits"]
    got = hits_to_numpy(a)[::97]
    for k in ("flags", "pType", "pIndex", "leafNode", "material"):
        assert np.array_equal(got[k], want[k]), k
    for k in ("t", "u", "v"):
        assert np.array_equal(bits(got[k]), bits(want[k])), k


def test_streams_are_reentrant(c3):
    torch = _torch()
    from tracer_b200 import rays_to_torch
    prim, scene, rays = c3
    d = rays_to_torch(rays[:1_000_000], "cuda:0")
    ref = scene.hit(d)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    outs = []
    for s in (s1, s2, s1, s2):
        with torch.cuda.stream(s):
            outs.append(scene.hit(d))
    torch.cuda.synchronize()
    for o in outs:
        assert torch.equal(o, ref)


def test_host_threads_are_reentrant(c3):
    """SURVEY 8b threading row: one immutable scene, several host threads tracing at once -- device-pointer calls on
    their own streams and host-pointer calls through the shared staging ring (ctypes drops the GIL inside the call)."""
    import threading
    torch = _torch()
    from tracer_b200 import hits_to_numpy, rays_to_torch
    prim, scene, rays = c3
    sub = np.ascontiguousarray(rays[:700_000])
    d = rays_to_torch(sub, "cuda:0")
    want = hits_to_numpy(scene.hit(d)).view(np.uint8)
    torch.cuda.synchronize()
    results, errors = {}, []

    def device_worker(k):
        try:
            st = torch.cuda.Stream()
            with torch.cuda.stream(st):
                outs = [scene.hit(d) for _ in range(6)]
            st.synchronize()
            results[k] = [hits_to_numpy(o).view(np.uint8) for o in outs]
        except Exception as e:                                   # noqa: BLE001
            errors.append(e)

    def host_worker(k):
        try:
            results[k] = [scene.hit(sub).view(np.uint8) for _ in range(3)]
        except Exception as e:                                   # noqa: BLE001
            errors.append(e)

    threads = [threading.Thread(target=device_worker, args=(k,)) for k in range(3)]
    threads += [threading.Thread(target=host_worker, args=(k,)) for k in (3, 4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for k, outs in results.items():
        for o in outs:
            assert np.array_equal(o.reshape(-1), want.reshape(-1)), f"thread {k}"


def test_sort_hint_changes_nothing_but_order_of_work(c3):
    """TRQ_SORT_RAYS reorders the work queue only: identical bytes out, for incoherent rays and for the degenerate
    batch whose rays all start at one point (one histogram bin)."""
    torch = _torch()
    from tracer_b200 import harness as H, rays_to_torch
    prim, scene, rays = c3
    d = rays_to_torch(rays[:2_000_000], "cuda:0")
    assert torch.equal(scene.hit(d, sort=True), scene.hit(d))
    assert torch.equal(scene.hit(d, any=True, sort=True), scene.hit(d, any=True))
    primary = rays_to_torch(H.cornell_camera_rays(1920, 1080), "cuda:0")
    assert torch.equal(scene.hit(primary, sort=True), scene.hit(primary))
    host = scene.hit(rays[:300_000].copy())
    assert np.array_equal(host.view(np.uint8), scene.hit(rays_to_torch(rays[:300_000], "cuda:0"), sort=True).cpu().numpy().view(np.uint8).reshape(-1))


def test_async_host_calls_equal_sync(c3):
    """TRQ_HOST_ASYNC: queued back-to-back calls through the shared staging ring give the bytes of the synchronous path."""
    torch = _torch()
    prim, scene, rays = c3
    sub = np.ascontiguousarray(rays[:1_500_000])
    want = scene.hit(sub)
    h_rays = torch.from_numpy(sub.view(np.float32).reshape(-1, 8)).pin_memory()
    outs = [torch.empty((sub.size, 8), dtype=torch.float32).pin_memory() for _ in range(3)]
    for o in outs:
        scene.hit_host(h_rays.data_ptr(), sub.size, o.data_ptr(), asynchronous=True)
    scene.host_sync()
    for o in outs:
        assert np.array_equal(o.numpy().view(np.uint8).reshape(-1), want.view(np.uint8).reshape(-1))


def test_c4_any_hit_full_scene(built, port):
    """BASELINE C4: C3 geometry + 10,012 sphere leaves, any-hit shadow rays toward the light squares with
    tmax = distance to the light sample; occlusion flag AND the primitive found are bit-exact (the traversal
    order is the reference's, so the first accepted hit is the same one)."""
    torch = _torch()
    from tracer_b200 import Scene, harness as H, hits_to_numpy, rays_to_torch
    prim = H.scene_c4(2)
    scene = Scene(prim, 0)
    assert scene.info["nSphere"] == 10_012 and scene.info["nTri"] > 1_000_000
    primary = H.cornell_camera_rays(1920, 1080)
    d = rays_to_torch(primary, "cuda:0")
    recs = scene.expand(d, scene.hit(d)).cpu().numpy().view(L.record_dtype).reshape(-1)
    la, lb = H.scene_c4_lights(prim)
    shadow, _ = H.shadow_rays(recs, la, lb, 0)
    assert shadow.size > 1_000_000
    ds = rays_to_torch(shadow, "cuda:0")
    a = scene.hit(ds, any=True)
    got = hits_to_numpy(a)
    naive = hits_to_numpy(scene.hit(ds, any=True, reflayout=True))
    for k in got.dtype.names:
        bad = np.nonzero(bits(got[k]) != bits(naive[k]))[0]
        assert bad.size == 0, f"packed vs reference-layout kernel: {k} differs on {bad.size} rays, first {bad[:4]}: {got[bad[:4]]} vs {naive[bad[:4]]}"
    occluded = (got["flags"] & 1) == 1
    assert 0.02 < occluded.mean() < 0.98                         # a real mix of lit and shadowed points
    assert bool((got["t"][occluded] < shadow["tmax"][occluded]).all())
    sub = np.ascontiguousarray(shadow[::23])
    want = port.trace(prim, sub, any=True, nthreads=8)["hits"]
    g = got[::23]
    for k in ("flags", "pType", "pIndex", "leafNode", "material"):
        assert np.array_equal(g[k], want[k]), k
    assert np.array_equal(bits(g["t"]), bits(want["t"]))
    # closest-hit over the same rays can only be nearer or equal, and agrees on occlusion
    c = hits_to_numpy(scene.hit(ds))
    assert np.array_equal(c["flags"] & 1, got["flags"] & 1)
    assert bool((c["t"][occluded] <= got["t"][occluded]).all())


def test_c1_sphere_scene_full_batch(built, port, capsys):
    """BASELINE C1: the 485-sphere randomScene as Sphere leaves, all 921,600 primary rays against the oracle: ids and t bit
    for bit, sphere uv (atan2f / asinf) inside CUDA's documented error of the float64 value (assert_sphere_uv), the
    oracle's bits at the poles -- where rounding pushes |gn.y| above 1 on the r = 1000 ground sphere, both sides give NaN."""
    _torch()
    from tracer_b200 import Scene, harness as H, hits_to_numpy, rays_to_torch
    from .test_gpu_parity import assert_hits_equal
    from .test_special_rays_cpu import sphere_uv_error
    prim = H.scene_c1()
    scene = Scene(prim, 0)
    rays = H.camera_rays((13, 2, 3), (0, 0, 0), np.float32(20 * np.pi / 180), 1280, 720)
    assert rays.size == 921_600
    got = hits_to_numpy(scene.hit(rays_to_torch(rays, "cuda:0")))
    want = port.trace(prim, rays, records=True, nthreads=8)
    assert_hits_equal(got, want["hits"], "c1", want["records"])
    sph = (want["hits"]["flags"] & 1) == 1
    assert (want["hits"]["pType"][sph] == L.SPHERE).all() and sph.sum() > 500_000
    eu, ev = sphere_uv_error(got["u"][sph], got["v"][sph], want["records"]["gn"][sph])
    with capsys.disabled():
        print(f"\nC1 full batch, sphere uv: largest error of phi (atan2f) {eu} ulp, of theta (asinf) {ev} ulp")
