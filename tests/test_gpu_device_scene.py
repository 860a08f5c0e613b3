"""GPU: the scene can be built, created and refitted without the tree ever visiting the host.

  trq_bvh_build_tree_device    BVH::buildTree (BVH.hh:246-269) with leaves and result in device memory
  trq_scene_create_device      validation + numbering of the reference-layout tree as kernels (kernels/plan_scene.cuh);
                               must give the layout trq_scene_create's host walk gives
  trq_scene_update_vertices    refit: triangle leaf boxes from the moved vertices (AAPLRenderer.mm:575-589), interior
                               boxes as unions of their children (BVH.hh:229-231)
"""
import ctypes as C
import time

import numpy as np
import pytest

from tracer_b200 import layout as L

from .test_gpu_parity import _torch, assert_like_oracle, gpu_trace
from .util import refit_on_host

pytestmark = pytest.mark.gpu


def _leaves(prim):
    n = int((prim.bvhList["pType"] != L.BVH).sum())
    return prim.bvhList[1:n + 1].copy() if prim.bvhList.size > 1 else prim.bvhList.copy()


def test_device_builder_matches_the_host_builder(built):
    torch = _torch()
    from tracer_b200 import BVHBuilder, harness as H
    for prim in (H.scene_soup(20000, seed=3, extent=0.05), H.scene_c2(), H.scene_reference_cornell()):
        b = BVHBuilder()
        b._chunks.append(_leaves(prim))
        dev = b.buildTreeDevice(0)
        got = dev.cpu().numpy().view(L.bvh_dtype).reshape(-1)
        assert np.array_equal(got.view(np.uint8), prim.bvhList.view(np.uint8)), "device-resident build differs from the host builder's tree"


def test_scene_created_on_the_device_equals_scene_created_from_the_host(built, port):
    torch = _torch()
    from tracer_b200 import DevicePrimitive, Scene, harness as H
    tri = H.make_vertices(np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], dtype=np.float32), [[0, 1, 2], [0, 1, 3]])
    cases = [
        (H.scene_reference_cornell(), H.cornell_camera_rays(320, 180), H.random_rays(100000, seed=5, lo=(-245, 0, 0), hi=(800, 555, 555))),
        (H.scene_soup(200000, seed=1, extent=0.01), H.random_rays(200000, seed=2), H.random_rays(50000, seed=3)),
        (H.scene_c1(), H.camera_rays((13, 2, 3), (0, 0, 0), np.float32(20 * np.pi / 180), 320, 180), H.random_rays(20000, seed=4, lo=(-5, 0, -5), hi=(5, 2, 5))),
        (H.build_primitive(tri, np.array([0, 1, 2], dtype=np.uint32)), H.random_rays(1000, seed=1, lo=(-0.5, -0.5, -0.5), hi=(1, 1, 1)), None),
        (H.build_primitive(tri, np.array([0, 1, 2, 0, 1, 3], dtype=np.uint32)), H.random_rays(1000, seed=2, lo=(-0.5, -0.5, -0.5), hi=(1, 1, 1)), None),
    ]
    for prim, rays_a, rays_b in cases:
        host = Scene(prim, 0)
        dev = Scene(DevicePrimitive.from_host(prim, "cuda:0"), 0)
        for k in ("nNode", "nInterior", "nLeaf", "maxDepth", "nTri", "nSphere", "nSquare", "nCube", "topNodes", "bytesPacked"):
            assert host.info[k] == dev.info[k], (k, host.info, dev.info)
        for rays, any_hit in ((rays_a, False), (rays_b, True)):
            if rays is None:
                continue
            a, b = gpu_trace(host, rays, any_hit), gpu_trace(dev, rays, any_hit)
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), "device-planned scene answers differently"
            assert_like_oracle(b, port, prim, rays, any_hit, "device-created scene")
        for c in range(len(Scene.kernel_configs())):           # the staged top-of-tree block must be the same block
            try:
                host.set_kernel_config(c); dev.set_kernel_config(c)
            except Exception:
                continue
            a, b = gpu_trace(host, rays_a), gpu_trace(dev, rays_a)
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), c
        host.close(); dev.close()


def test_device_validation_reports_what_the_host_walk_reports(built):
    torch = _torch()
    from tracer_b200 import DevicePrimitive, Scene, harness as H
    from tracer_b200._lib import ERR_LAYOUT, TrqError
    from tracer_b200.scene import Primitive
    prim = H.scene_soup(500, seed=1, extent=0.2)

    def broken(mut):
        b = prim.bvhList.copy()
        mut(b)
        return Primitive(triList=prim.triList, idxList=prim.idxList, bvhList=b)

    leaf = int(np.nonzero(prim.bvhList["pType"] == L.TRIANGLE)[0][0])
    inner = int(np.nonzero(prim.bvhList["pType"] == L.BVH)[0][1])
    muts = [lambda b: b["left"].__setitem__(0, b.size + 5),                 # child index out of range
            lambda b: b["right"].__setitem__(0, b["left"][0]),               # not a tree
            lambda b: b["pIndex"].__setitem__(leaf, 10 ** 6),                # primitive index out of range
            lambda b: b["parent"].__setitem__(inner, inner),                 # parent link does not point back
            lambda b: b["parent"].__setitem__(0, 3)]                         # root's parent
    for mut in muts:
        bad = broken(mut)
        with pytest.raises(TrqError) as e_host:
            Scene(bad, 0)
        with pytest.raises(TrqError) as e_dev:
            Scene(DevicePrimitive.from_host(bad, "cuda:0"), 0)
        assert e_host.value.status == ERR_LAYOUT and e_dev.value.status == ERR_LAYOUT
    Scene(DevicePrimitive.from_host(prim, "cuda:0"), 0).close()          # and the GPU is still healthy


def test_build_and_create_without_leaving_the_gpu(built, port):
    """1 M-triangle class scene: leaves -> tree -> scene, all in device memory; wall time reported."""
    torch = _torch()
    from tracer_b200 import BVHBuilder, DevicePrimitive, Scene, harness as H
    prim = H.scene_soup(300000, seed=7, extent=0.01)
    b = BVHBuilder()
    b._chunks.append(_leaves(prim))
    tri = torch.from_numpy(prim.triList.view(np.uint8).reshape(-1).copy()).cuda()
    idx = torch.from_numpy(prim.idxList.view(np.uint8).reshape(-1).copy()).cuda()
    for rep in range(3):                                       # first call pays for the scratch pool
        torch.cuda.synchronize(); t0 = time.perf_counter()
        nodes = b.buildTreeDevice(0)
        t1 = time.perf_counter()
        scene = Scene(DevicePrimitive(triList=tri, idxList=idx, bvhList=nodes), 0)
        torch.cuda.synchronize(); t2 = time.perf_counter()
        print(f"device build {1e3 * (t1 - t0):.2f} ms + create {1e3 * (t2 - t1):.2f} ms for {prim.nTri} triangles")
        if rep < 2:
            scene.close()
    assert np.array_equal(nodes.cpu().numpy().view(L.bvh_dtype).reshape(-1).view(np.uint8), prim.bvhList.view(np.uint8))
    rays = H.random_rays(200000, seed=2)
    assert_like_oracle(gpu_trace(scene, rays), port, prim, rays, False, "built + created on the device")
    scene.close()


def test_refit_after_the_vertices_moved(built, port):
    torch = _torch()
    from tracer_b200 import Scene, harness as H
    for prim, rays in ((H.scene_soup(20000, seed=5, extent=0.05), H.random_rays(100000, seed=8)),
                       (H.scene_reference_cornell(), H.cornell_camera_rays(320, 180))):
        scene = Scene(prim, 0)
        rng = np.random.default_rng(1)
        verts = prim.triList.copy()
        verts["v"] += (rng.random(verts["v"].shape, dtype=np.float32) - np.float32(0.5)) * np.float32(0.02) * np.abs(verts["v"]).max()
        moved = refit_on_host(prim, verts)
        for how in ("host", "device"):
            scene.update_vertices(verts if how == "host" else torch.from_numpy(verts.view(np.uint8).reshape(-1).copy()).cuda())
            for any_hit in (False, True):
                assert_like_oracle(gpu_trace(scene, rays, any_hit), port, moved, rays, any_hit, f"refit ({how})")
            for c in range(len(Scene.kernel_configs())):
                try:
                    scene.set_kernel_config(c)
                except Exception:
                    continue
                assert_like_oracle(gpu_trace(scene, rays), port, moved, rays, False, f"refit cfg {c}")
            scene.set_kernel_config(-1)
        scene.update_vertices(prim.triList)                     # and back: the original answers return
        assert_like_oracle(gpu_trace(scene, rays), port, prim, rays, False, "refit back")
        scene.close()
