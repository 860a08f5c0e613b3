"""GPU: every launch configuration of the traversal kernel (CTA size x CTAs per SM; top of the tree staged in shared
memory by TMA bulk copies or not) and both record formats (trq_hit, trq_hit16) produce the oracle's results.

The top-of-tree block is the first `topNodes` packed interior nodes in breadth-first order; a configuration stages a
prefix of it, so the residency test inside the kernel is "index < topCount" (Render.hh:145-160 re-reads those levels
from memory for every ray)."""
import numpy as np
import pytest

from tracer_b200 import layout as L

from .test_gpu_parity import _torch, assert_hits_equal, assert_like_oracle, gpu_trace, oracle

pytestmark = pytest.mark.gpu


def _configs():
    from tracer_b200 import Scene
    return list(enumerate(Scene.kernel_configs()))


def test_every_configuration_matches_the_oracle(built, port):
    torch = _torch()
    from tracer_b200 import Scene, harness as H
    names = Scene.kernel_configs()
    assert len(names) >= 2 and "top=false" in names[0] and any("top=true" in n for n in names)
    soup = H.scene_soup(200000, seed=1, extent=0.01)
    mixed = H.scene_reference_cornell()
    cases = [(soup, H.random_rays(300000, seed=2), False), (soup, H.random_rays(100000, seed=3), True),
             (mixed, H.cornell_camera_rays(320, 180), False),
             (mixed, H.random_rays(100000, seed=5, lo=(-245, 0, 0), hi=(800, 555, 555)), True)]
    wants = [oracle(port, p, r, a) for p, r, a in cases]
    staged_any = False
    for prim in (soup, mixed):
        scene = Scene(prim, 0)
        assert 0 < scene.info["topNodes"] <= min(2047, scene.info["nInterior"])
        for c, name in enumerate(names):
            try:
                staged = scene.set_kernel_config(c)
            except Exception:                                  # a configuration may not fit a deep tree
                continue
            assert (staged > 0) == ("top=true" in name), (name, staged)
            staged_any |= staged > 0
            for (p, rays, any_hit), want in zip(cases, wants):
                if p is prim:
                    assert_hits_equal(gpu_trace(scene, rays, any_hit), want[0], f"cfg {name}", want[1])
        scene.close()
    assert staged_any
    # the library's own choice: staging only for trees that fit into the staged block whole
    small, mid, big = Scene(H.scene_c1(), 0), Scene(mixed, 0), Scene(soup, 0)
    assert small.set_kernel_config(-1) == small.info["nInterior"] and "top=true" in small.kernel_config()
    assert mid.set_kernel_config(-1) == 0 and big.set_kernel_config(-1) == 0 and "top=false" in big.kernel_config()
    small.close(); mid.close(); big.close()


def test_hit16_is_the_packed_form_of_trq_hit(built, port):
    torch = _torch()
    from tracer_b200 import Scene, harness as H, rays_to_torch
    for prim, rays in ((H.scene_reference_cornell(), H.cornell_camera_rays(320, 180)),
                       (H.scene_soup(100000, seed=4, extent=0.02), H.random_rays(200000, seed=6))):
        scene = Scene(prim, 0)
        d = rays_to_torch(rays, "cuda:0")
        for any_hit in (False, True):
            full = scene.hit(d, any=any_hit).cpu().numpy().view(L.hit_dtype).reshape(-1)
            for c in range(len(Scene.kernel_configs())):
                try:
                    scene.set_kernel_config(c)
                except Exception:
                    continue
                small = scene.hit(d, any=any_hit, hit16=True)
                assert small.shape == (rays.size, 4)
                got = small.cpu().numpy().view(L.hit16_dtype).reshape(-1)
                assert np.array_equal(got.view(np.uint8), L.pack_hit16(full).view(np.uint8)), (c, any_hit)
            scene.set_kernel_config(-1)
        # host-pointer path with 16-byte records (half the D2H bytes)
        host = scene.hit(rays, hit16=True)
        assert host.dtype == L.hit16_dtype
        want = port.trace(prim, rays, nthreads=8)["hits"]
        assert np.array_equal(host["id"], L.pack_hit16(want)["id"])
        assert np.array_equal(host["t"].view(np.uint32), want["t"].view(np.uint32))
        scene.close()


def test_host_path_chunk_boundaries(built):
    """TRQ_HOST_PTRS cuts a large batch into chunks that cycle through four staging buffers; every ray must land at its own
    index for sizes around the chunk boundaries, for both record formats."""
    import os
    torch = _torch()
    from tracer_b200 import Scene, harness as H, rays_to_torch
    prim = H.scene_soup(50000, seed=9, extent=0.03)
    scene = Scene(prim, 0)
    os.environ["TRQ_CHUNK_RAYS"] = "16384"
    try:
        for n in (16384 * 6, 16384 * 6 + 1, 16384 * 9 + 777, 16384 * 5 + 3, 1000):
            rays = H.random_rays(n, seed=n % 97)
            dev = scene.hit(rays_to_torch(rays, "cuda:0")).cpu().numpy().view(L.hit_dtype).reshape(-1)
            for h16 in (False, True):
                host = scene.hit(rays, hit16=h16)
                want = L.pack_hit16(dev) if h16 else dev
                assert np.array_equal(host.view(np.uint8), want.view(np.uint8)), (n, h16)
    finally:
        del os.environ["TRQ_CHUNK_RAYS"]
    scene.close()


def test_automatic_ray_ordering(built, port):
    """Without TRQ_SORT_RAYS, a scene whose tree is much larger than L2 has large batches examined on the device: incoherent
    ones are ordered before the traversal, coherent ones are left as given. TRQ_AUTO_SORT=1 applies the rule to a small
    scene here. Whatever it decides, every ray's record lands at the ray's own index and equals the unordered result."""
    import os
    torch = _torch()
    from tracer_b200 import Scene, harness as H, rays_to_torch
    prim = H.scene_soup(100000, seed=21, extent=0.02)
    scene = Scene(prim, 0)
    n = (1 << 20) + 12345
    incoherent = H.random_rays(n, seed=4)
    coherent = np.repeat(H.camera_rays((0.5, 0.5, -2.0), (0.5, 0.5, 0.5), np.float32(0.6), 1280, 720), 2)[:n]   # neighbours share cell and octant
    os.environ["TRQ_AUTO_SORT"] = "1"
    try:
        for rays in (incoherent, coherent):
            d = rays_to_torch(np.ascontiguousarray(rays), "cuda:0")
            plain = scene.hit(d, sort=False).clone()                 # TRQ_NO_SORT
            for any_hit in (False, True):
                ref = scene.hit(d, any=any_hit, sort=False).clone()
                auto = scene.hit(d, any=any_hit)                       # the library decides
                hinted = scene.hit(d, any=any_hit, sort=True)
                assert torch.equal(auto.view(torch.int32), ref.view(torch.int32))
                assert torch.equal(hinted.view(torch.int32), ref.view(torch.int32))
            sub = np.arange(0, rays.size, 97)
            assert_like_oracle(plain.cpu().numpy().view(L.hit_dtype).reshape(-1)[sub], port, prim, np.ascontiguousarray(rays[sub]),
                               False, "auto ordering")
    finally:
        del os.environ["TRQ_AUTO_SORT"]
    scene.close()
