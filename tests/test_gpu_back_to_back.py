"""GPU: traces issued back to back on one stream, with no synchronisation between the calls, give what separate
synchronous traces give, byte for byte. A trace that follows another trace of the same (unchanged) tree is an early
launch: its CTAs start while the previous kernel on the stream still runs, trace the rays they drew first, and check
those rays again once that kernel has finished. The cases below are the ones where what an early CTA read first can be
stale: the same output buffer, rays rewritten by a caller's kernel or by the previous trace itself, a refit in between,
and graph replays (captured launches are never early) between eager ones."""
import numpy as np
import pytest

from .test_gpu_parity import _torch

pytestmark = pytest.mark.gpu

_scenes = {}


def _scene(kind):
    """(Scene, incoherent rays inside it as a CUDA tensor): the C3 meshes scene (~1 M triangles) or a small soup."""
    if kind not in _scenes:
        from tracer_b200 import Scene, harness as H, rays_to_torch
        if kind == "c3":
            prim, n, lo, hi = H.scene_c3(2), 1 << 20, (0, 0, 0), (555, 555, 555)
        else:
            prim, n, lo, hi = H.scene_soup(20000, seed=3, extent=0.05), 70000, (0, 0, 0), (1, 1, 1)
        rays = [rays_to_torch(H.random_rays(n, seed=40 + k, lo=lo, hi=hi), "cuda:0") for k in range(2)]
        _scenes[kind] = (prim, Scene(prim, 0), rays)
    return _scenes[kind]


def _sync_hit(torch, scene, rays, **kw):
    torch.cuda.synchronize()
    out = scene.hit(rays, **kw).clone()
    torch.cuda.synchronize()
    return out


def _eq(torch, got, want, what):
    assert torch.equal(got.view(torch.int32), want.view(torch.int32)), what


@pytest.mark.parametrize("kind", ["small", "c3"])
@pytest.mark.parametrize("any_hit", [False, True])
@pytest.mark.parametrize("hit16", [False, True])
def test_two_batches_into_one_buffer(built, kind, any_hit, hit16):
    torch = _torch()
    _, scene, (a, b) = _scene(kind)
    want_a = _sync_hit(torch, scene, a, any=any_hit, hit16=hit16)
    want_b = _sync_hit(torch, scene, b, any=any_hit, hit16=hit16)
    out, other = torch.empty_like(want_a), torch.empty_like(want_a)
    scene.hit(a, any=any_hit, hit16=hit16, out=out)
    scene.hit(b, any=any_hit, hit16=hit16, out=out)          # the second writes over the first
    scene.hit(a, any=any_hit, hit16=hit16, out=other)
    scene.hit(a, any=any_hit, hit16=hit16, out=out)
    scene.hit(b, any=any_hit, hit16=hit16, out=out)
    torch.cuda.synchronize()
    _eq(torch, out, want_b, "last batch into the shared buffer")
    _eq(torch, other, want_a, "batch between two others")


@pytest.mark.parametrize("kind", ["small", "c3"])
def test_rays_rewritten_by_a_kernel_between_traces(built, kind):
    torch = _torch()
    _, scene, (a, b) = _scene(kind)
    mixed = a.clone()
    mixed[::3] = b[::3]                                      # every third ray changes, the others stay
    want_a = _sync_hit(torch, scene, a)
    want_mixed = _sync_hit(torch, scene, mixed)
    rays = a.clone()
    o1, o2, o3 = torch.empty_like(want_a), torch.empty_like(want_a), torch.empty_like(want_a)
    torch.cuda.synchronize()
    scene.hit(rays, out=o1)
    torch.bitwise_or(mixed.view(torch.int32), 0, out=rays.view(torch.int32))     # one elementwise kernel writes the rays
    scene.hit(rays, out=o2)
    scene.hit(rays, out=o3)
    torch.cuda.synchronize()
    _eq(torch, o1, want_a, "before the rewrite")
    _eq(torch, o2, want_mixed, "right after the rewriting kernel")
    _eq(torch, o3, want_mixed, "after that")


@pytest.mark.parametrize("kind", ["small", "c3"])
def test_rays_alias_the_previous_hit_buffer(built, kind):
    """The second call's rays are the first call's output buffer, which held other valid rays before the first call."""
    torch = _torch()
    _, scene, (a, b) = _scene(kind)
    want_a = _sync_hit(torch, scene, a)
    want_aa = _sync_hit(torch, scene, want_a)                  # hit records read as rays
    buf = b.clone()
    out = torch.empty_like(want_a)
    torch.cuda.synchronize()
    scene.hit(a, out=buf)
    scene.hit(buf, out=out)
    torch.cuda.synchronize()
    _eq(torch, buf, want_a, "first trace")
    _eq(torch, out, want_aa, "trace of the first one's output")


def test_update_vertices_between_traces(built):
    torch = _torch()
    from tracer_b200 import Scene, harness as H, rays_to_torch
    prim = H.scene_c2()
    scene = Scene(prim, 0)
    rays = rays_to_torch(H.cornell_camera_rays(320, 180), "cuda:0")
    want_before = _sync_hit(torch, scene, rays)
    moved = prim.triList.copy()
    rng = np.random.default_rng(5)
    moved["v"] += rng.uniform(-2.0, 2.0, moved["v"].shape).astype(np.float32)
    o1, o2, o3 = (torch.empty_like(want_before) for _ in range(3))
    scene.hit(rays, out=o1)
    scene.hit(rays, out=o1)
    scene.update_vertices(moved)
    scene.hit(rays, out=o2)
    scene.hit(rays, out=o3)
    torch.cuda.synchronize()
    want_after = _sync_hit(torch, scene, rays, reflayout=True)
    assert not torch.equal(want_after.view(torch.int32), want_before.view(torch.int32))
    _eq(torch, o1, want_before, "before the update")
    _eq(torch, o2, want_after, "first trace after the update")
    _eq(torch, o3, want_after, "second trace after the update")
    scene.close()


def test_captured_two_trace_graph_between_eager_traces(built):
    torch = _torch()
    _, scene, (a, b) = _scene("small")
    want_a = _sync_hit(torch, scene, a)
    want_b_any = _sync_hit(torch, scene, b, any=True)
    side = torch.cuda.Stream()
    g1, g2, e1, e2 = (torch.empty_like(want_a) for _ in range(4))
    with torch.cuda.stream(side):
        scene.hit(a, out=g1)                                   # warm the stream before capture
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            scene.hit(a, out=g1)
            scene.hit(b, any=True, out=g2)
        for rep in range(3):
            for t in (g1, g2, e1, e2):
                t.zero_()
            scene.hit(b, any=True, out=e1)
            g.replay()
            scene.hit(a, out=e2)
            g.replay()
            torch.cuda.synchronize()
            _eq(torch, g1, want_a, f"replay {rep}: first trace")
            _eq(torch, g2, want_b_any, f"replay {rep}: second trace")
            _eq(torch, e1, want_b_any, f"replay {rep}: eager before")
            _eq(torch, e2, want_a, f"replay {rep}: eager between")
