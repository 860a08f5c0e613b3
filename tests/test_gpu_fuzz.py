"""GPU: randomized parity sweep aimed at the places where CUDA and host arithmetic could part ways: rays with zero
direction components (1/0 = inf slabs), origins lying exactly on box planes / vertices / edges (0 * inf = NaN inside
AABB::hit_t, where only fminf/fmaxf's NaN rule decides), degenerate and duplicated triangles, tiny and huge tmax,
mixed leaf types, any-hit and closest-hit, both kernels."""
import os

import numpy as np
import pytest

from tracer_b200 import layout as L

from .test_gpu_parity import assert_hits_equal, gpu_trace

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def adversarial_rays(rng, prim, n):
    from tracer_b200._lib import lib
    bvh = prim.bvhList
    rays = np.zeros(n, dtype=L.ray_dtype)
    lo, hi = bvh["mini"][0], bvh["maxi"][0]
    rays["o"] = rng.uniform(lo - 0.2 * (hi - lo) - 1e-3, hi + 0.2 * (hi - lo) + 1e-3, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    k = np.arange(n)
    d[k % 4 == 1, rng.integers(3)] = 0.0                                   # one zero component
    two = k % 16 == 2
    d[two] = 0.0; d[two, rng.integers(3)] = rng.choice([-1.0, 1.0])        # axis-aligned
    # origins exactly on a plane of some node's box, on a vertex, or on an edge midpoint
    node = bvh[rng.integers(0, bvh.size, n)]
    plane = k % 3 == 0
    ax = rng.integers(0, 3, n)
    on = np.where(rng.random(n) < 0.5, node["mini"][k, ax], node["maxi"][k, ax])
    rays["o"][plane, ax[plane]] = on[plane]
    if prim.triList.size:
        v = prim.triList["v"]
        tri = prim.idxList.reshape(-1, 3)[rng.integers(0, prim.nTri, n)]
        vert = k % 7 == 3
        rays["o"][vert] = v[tri[vert, 0]]
        edge = k % 7 == 5
        target = (v[tri[edge, 0]] + v[tri[edge, 1]]) * np.float32(0.5)     # aim exactly at an edge midpoint
        d[edge] = target - rays["o"][edge]
    rays["d"] = d
    lib.trqh_normalize_rays(rays.ctypes.data, n)
    bad = ~np.isfinite(rays["d"]).all(axis=1)                              # 0/0 from a zero-length direction
    rays["d"][bad] = np.array([0, 0, 1], dtype=np.float32)
    tm = np.full(n, L.FLT_MAX, dtype=np.float32)
    tm[k % 5 == 0] = rng.uniform(1e-3, 3.0, (k % 5 == 0).sum()).astype(np.float32) * np.float32(np.linalg.norm(hi - lo))
    tm[k % 11 == 0] = np.float32(1e-30)
    rays["tmax"] = tm
    return rays


def scenes(rng):
    from tracer_b200 import harness as H
    yield "cornell mixed", H.scene_reference_cornell()
    yield "soup", H.scene_soup(3000, seed=int(rng.integers(1 << 30)), extent=0.15)
    # degenerate + duplicated + axis-aligned triangles on an integer lattice (many exact ties, flat boxes)
    pts = rng.integers(-3, 4, (600, 3, 3)).astype(np.float32)
    pts[::9, 2] = pts[::9, 1]                                              # zero-area triangles
    pts[1::13] = pts[0::13][: len(pts[1::13])]                             # exact duplicates
    ms = H.MeshSoup()
    for t in pts:
        ms.add(t, [[0, 1, 2]])
    tri, idx = ms.arrays()
    yield "lattice", H.build_primitive(tri, idx)
    sph = np.array([H.make_sphere(float(rng.uniform(0.2, 1.5)), rng.uniform(-3, 3, 3), i) for i in range(60)], dtype=L.sphere_dtype)
    yield "spheres", H.build_primitive(spheres=sph)
    # cubes whose model matrices scale down / up / shear-free rotate, spheres and squares around them: the leaf types whose
    # records the packed kernel finishes out of line
    cubes = []
    for i in range(6):
        sc = rng.uniform(0.01, 0.05, 3) if i % 2 == 0 else rng.uniform(0.5, 2.0, 3)
        m = H.translation4x4(*rng.uniform(-3, 3, 3)) @ H.rotation4x4(float(rng.uniform(0, 3)), (0, 1, 0)) @ H.scale4x4(*sc)
        c = H.make_cube(m, i)
        if i % 2 == 0:
            c["box_mini"], c["box_maxi"] = (-50, -40, -30), (50, 40, 30)
        cubes.append(c)
    yield "cubes", H.build_primitive(cubes=np.array(cubes, dtype=L.cube_dtype), spheres=sph[:10])


def _seeds():
    """Three seeds in the regular suite; TRQ_FUZZ_SEEDS=lo-hi widens the campaign (profiles/r01_fuzz_campaign.txt)."""
    extra = os.environ.get("TRQ_FUZZ_SEEDS", "")
    if "-" in extra:
        lo, hi = (int(x) for x in extra.split("-"))
        return [1, 2, 3] + list(range(lo, hi + 1))
    return [1, 2, 3]


def _assert_records(scene, rays, hits_dev, want, where):
    """trq_expand_hits on adversarial rays: the HitRecord fields of every hit, bit for bit (sphere uv: libm vs CUDA)."""
    from tracer_b200 import rays_to_torch
    recs = scene.expand(rays_to_torch(rays, f"cuda:{scene.device}"), hits_dev).cpu().numpy().view(L.record_dtype).reshape(-1)
    w = want["records"]
    assert np.array_equal(recs["hit"], w["hit"]), where
    m = w["hit"] == 1
    sph = want["hits"]["pType"] == L.SPHERE
    for k in ("t", "p", "gn", "sn", "front", "material"):
        a, b = recs[k][m].view(np.uint32), w[k][m].view(np.uint32)
        # a NaN component (0 * inf in a degenerate hit) has no agreed payload: compare NaN-ness there, bits elsewhere
        if recs[k].dtype.kind == "f":
            na, nb = np.isnan(recs[k][m]), np.isnan(w[k][m])
            assert np.array_equal(na, nb) and np.array_equal(a[~na], b[~nb]), f"{where}: {k}"
        else:
            assert np.array_equal(a, b), f"{where}: {k}"
    e = m & ~sph
    na = np.isnan(w["uv"][e])
    assert np.array_equal(np.isnan(recs["uv"][e]), na) and np.array_equal(recs["uv"][e].view(np.uint32)[~na], w["uv"][e].view(np.uint32)[~na]), f"{where}: uv"


@pytest.mark.parametrize("seed", _seeds())
def test_adversarial_parity(built, port, seed):
    """Every launch configuration of the packed kernel (it finishes the records of all five leaf types itself), both record
    formats, the reference-layout kernel and the HitRecord expansion, on the adversarial rays."""
    torch = _torch()
    from tracer_b200 import Scene, rays_to_torch
    rng = np.random.default_rng(seed)
    ncfg = len(Scene.kernel_configs())
    for name, prim in scenes(rng):
        scene = Scene(prim, 0)
        rays = adversarial_rays(rng, prim, 40000)
        d = rays_to_torch(rays, "cuda:0")
        for any_hit in (False, True):
            want = port.trace(prim, rays, any=any_hit, counters=True, records=True, nthreads=8)
            got = gpu_trace(scene, rays, any_hit, True)
            assert_hits_equal(got, want["hits"], f"{name} seed={seed} any={any_hit} reflayout", want["records"])
            for c in range(ncfg):
                try:
                    scene.set_kernel_config(c)
                except Exception:                              # a staged configuration may not fit a deep tree
                    continue
                where = f"{name} seed={seed} any={any_hit} cfg={c}"
                h = scene.hit(d, any=any_hit)
                got = h.cpu().numpy().view(L.hit_dtype).reshape(-1)
                assert_hits_equal(got, want["hits"], where, want["records"])
                h16 = scene.hit(d, any=any_hit, hit16=True).cpu().numpy().view(L.hit16_dtype).reshape(-1)
                assert np.array_equal(h16.view(np.uint8), L.pack_hit16(got).view(np.uint8)), where + " hit16"
                if not any_hit and c == 0:
                    _assert_records(scene, rays, h, want, where)
            scene.set_kernel_config(-1)
        scene.close()
