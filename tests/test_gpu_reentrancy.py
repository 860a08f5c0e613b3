"""GPU: trq_trace is re-entrant -- many launches in flight on many streams, and thousands of launches of mixed kinds on
one scene, more than the queue-head ring holds. Every eager launch draws its own work-queue head and the kernel's last CTA
re-arms it, so a head is zero whenever a launch picks it up -- whatever kind of launch used it before (round-1 regression:
heads left dirty by one kernel variant made the next variant skip rays; graph replays: tests/test_gpu_work_queue.py)."""
import threading

import numpy as np
import pytest

from tracer_b200 import layout as L

from .test_gpu_parity import _torch

pytestmark = pytest.mark.gpu


def test_512_launches_in_flight_on_8_streams(built):
    torch = _torch()
    from tracer_b200 import Scene, harness as H, rays_to_torch
    prim = H.scene_soup(100000, seed=1, extent=0.02)
    scene = Scene(prim, 0)
    sizes = [50000, 1, 333, 20000, 4097, 65536, 31, 9999]
    batches = [rays_to_torch(H.random_rays(n, seed=100 + k), "cuda:0") for k, n in enumerate(sizes)]
    want = [scene.hit(b).clone() for b in batches]
    want_any = [scene.hit(b, any=True).clone() for b in batches]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream() for _ in range(8)]
    outs = []
    for rep in range(64):                                      # 8 x 64 = 512 launches queued without a single synchronise
        for k, st in enumerate(streams):
            j = (k + rep) % len(batches)
            any_hit = (rep + k) % 3 == 0
            o = torch.empty_like(batches[j])
            scene.hit(batches[j], any=any_hit, out=o, stream=st.cuda_stream)
            outs.append((j, any_hit, o))
    torch.cuda.synchronize()
    for j, any_hit, o in outs:
        assert torch.equal(o.view(torch.int32), (want_any if any_hit else want)[j].view(torch.int32))
    scene.close()


def test_more_launches_than_queue_heads_and_mixed_kernels(built):
    """> 4096 launches (the ring wraps), alternating closest / any / 16-byte records / the reference-layout kernel."""
    torch = _torch()
    from tracer_b200 import Scene, harness as H, rays_to_torch
    prim = H.scene_soup(20000, seed=2, extent=0.05)
    scene = Scene(prim, 0)
    d = rays_to_torch(H.random_rays(3000, seed=5), "cuda:0")
    want = {(a, h): scene.hit(d, any=a, hit16=h).clone() for a in (False, True) for h in (False, True)}
    ref = scene.hit(d, reflayout=True).clone()
    assert torch.equal(ref.view(torch.int32), want[(False, False)].view(torch.int32))
    out32, out16 = torch.empty_like(want[(False, False)]), torch.empty_like(want[(False, True)])
    for k in range(4500):
        a, h = bool(k & 1), bool(k & 2)
        o = scene.hit(d, any=a, hit16=h, out=out16 if h else out32)
        if k % 500 == 499 or k > 4090:
            assert torch.equal(o.view(torch.int32), want[(a, h)].view(torch.int32)), k
        if k % 1000 == 0:
            scene.hit(d, reflayout=True, out=out32)
    scene.close()


def test_host_threads_share_one_scene(built):
    torch = _torch()
    from tracer_b200 import Scene, harness as H, rays_to_torch
    prim = H.scene_soup(50000, seed=3, extent=0.03)
    scene = Scene(prim, 0)
    scene.profile(True)                                        # the profiling ring is shared state too
    batches = [rays_to_torch(H.random_rays(20000 + 1000 * k, seed=k), "cuda:0") for k in range(4)]
    want = [scene.hit(b).clone() for b in batches]
    torch.cuda.synchronize()
    errors = []

    def worker(k):
        try:
            torch.cuda.set_device(0)
            st = torch.cuda.Stream()
            o = torch.empty_like(batches[k])
            for _ in range(100):
                scene.hit(batches[k], out=o, stream=st.cuda_stream)
            st.synchronize()
            if not torch.equal(o.view(torch.int32), want[k].view(torch.int32)):
                errors.append(k)
        except Exception as e:                                 # pragma: no cover
            errors.append(repr(e))

    ts = [threading.Thread(target=worker, args=(k,)) for k in range(4)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errors, errors
    n, a, b = scene.profile_read()
    assert 0 < n <= 64 and a > 0
    scene.profile(False)
    scene.close()


def test_wavefront_step_is_cuda_graph_capturable(built):
    """cast -> trace -> spawn -> trace_indirect issue nothing but kernels and stream-ordered allocations, so a whole
    wavefront step can be captured once and replayed (the reference re-encodes its command buffer every frame,
    AAPLRenderer.mm:712-720). Replays give the eager results bit for bit; any-hit and TRQ_SORT_RAYS launches capture too."""
    torch = _torch()
    from tracer_b200 import Scene, harness as H, rays_to_torch
    prim = H.scene_c2()
    scene = Scene(prim, 0)
    W, Hh = 320, 180
    cam = ((278, 278, -800), (278, 278, 278), (0, 1, 0), np.float32(45 * (np.pi / 180)))
    dev = "cuda:0"
    r0 = torch.empty((W * Hh, 8), dtype=torch.float32, device=dev); h0 = torch.empty_like(r0)
    r1 = torch.empty_like(r0); h1 = torch.zeros_like(r0); ha = torch.empty_like(r0)
    s1 = torch.empty(W * Hh, dtype=torch.int32, device=dev); c1 = torch.zeros(1, dtype=torch.int64, device=dev)
    big = rays_to_torch(H.random_rays(70000, seed=8, lo=(0, 0, 0), hi=(555, 555, 555)), dev); hs = torch.empty_like(big)

    def step():
        scene.cast_rays(*cam, W, Hh, out=r0)
        scene.hit(r0, out=h0)
        scene.spawn_bounce(r0, h0, seed_base=7, out=r1, src=s1, count=c1)
        scene.hit_indirect(r1, c1, out=h1)
        scene.hit(r0, any=True, out=ha)
        scene.hit(big, out=hs, sort=True)

    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        step()
    torch.cuda.synchronize()
    n1 = int(c1.item())
    assert 0 < n1 <= W * Hh
    # the bounce wave is compacted with one atomic per warp: its order varies from run to run, its content does not
    def canon():
        k = torch.argsort(s1[:n1].to(torch.int64))
        return [h0.clone(), h1[:n1][k].clone(), ha.clone(), hs.clone(), c1.clone()]
    want = canon()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        step()
    for rep in range(3):
        for t in (h0, h1, ha, hs):
            t.zero_()
        g.replay()
        torch.cuda.synchronize()
        for a, b in zip(want, canon()):
            assert torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a, b.view(torch.int32) if b.dtype == torch.float32 else b), rep
    scene.close()
