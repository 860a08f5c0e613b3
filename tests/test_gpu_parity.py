"""GPU parity: the CUDA path (through the C-ABI) against the CPU oracle on identical rays.

Bar (BASELINE.json north_star): hit flags and primitive ids bit-exact; t / barycentrics within 1e-5
relative -- we assert BIT-EXACT t/u/v for triangle, square and cube hits (same arithmetic order, no
FMA). Sphere uv comes from atan2f / asinf, which differ from libm by ulps: it must lie inside the interval that
CUDA's documented error bounds give around the float64 value (test_special_rays_cpu.assert_sphere_uv), which
needs the oracle's shading normals.
"""
import numpy as np
import pytest

from tracer_b200 import layout as L

from .test_special_rays_cpu import assert_sphere_uv

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def assert_hits_equal(got, want, where="", records=None):
    """trq_hit against the oracle's hits `want`: ids, flags, t, and u / v of non-sphere hits bit for bit; sphere uv by
    assert_sphere_uv against records["gn"] (port.trace(..., records=True)["records"] of the same rays), required when
    the oracle reports a sphere hit."""
    assert got.size == want.size
    for k in ("flags", "pType", "pIndex", "leafNode", "material"):
        bad = np.nonzero(got[k] != want[k])[0]
        assert bad.size == 0, f"{where}: {k} differs on {bad.size} rays, first {bad[:5]}: got {got[k][bad[:5]]} want {want[k][bad[:5]]}"
    bad = np.nonzero(got["t"].view(np.uint32) != want["t"].view(np.uint32))[0]
    assert bad.size == 0, f"{where}: t differs on {bad.size} rays"
    hit = (want["flags"] & 1) == 1
    sph = hit & (want["pType"] == L.SPHERE)
    exact = hit & ~sph
    for k in ("u", "v"):
        assert np.array_equal(got[k][exact].view(np.uint32), want[k][exact].view(np.uint32)), f"{where}: {k} not bit-exact"
    if sph.any():
        assert records is not None, f"{where}: {int(sph.sum())} sphere hits: pass the oracle's records to check their uv"
        assert records.size == want.size, f"{where}: records of other rays"
        assert_sphere_uv(got["u"][sph], got["v"][sph], records["gn"][sph], want["u"][sph], want["v"][sph], where)


def oracle(port, prim, rays, any=False):
    """-> (hits, records) of the oracle for `rays`: what assert_hits_equal needs."""
    w = port.trace(prim, rays, any=any, records=True, nthreads=8)
    return w["hits"], w["records"]


def assert_like_oracle(got, port, prim, rays, any=False, where=""):
    """assert_hits_equal against the oracle's hits and records for `rays`."""
    want, records = oracle(port, prim, rays, any)
    assert_hits_equal(got, want, where, records)


def gpu_trace(scene, rays, any=False, reflayout=False, host=False):
    torch = _torch()
    from tracer_b200 import hits_to_numpy, rays_to_torch
    if host:
        return scene.hit(rays, any=any, reflayout=reflayout)
    d = rays_to_torch(rays, f"cuda:{scene.device}")
    h = scene.hit(d, any=any, reflayout=reflayout)
    torch.cuda.synchronize()
    return hits_to_numpy(h)


@pytest.fixture(scope="module")
def c2(built):
    _torch()
    from tracer_b200 import Scene, harness as H
    prim = H.scene_c2()
    return prim, Scene(prim, 0)


@pytest.fixture(scope="module")
def refcornell(built):
    _torch()
    from tracer_b200 import Scene, harness as H
    prim = H.scene_reference_cornell()
    return prim, Scene(prim, 0)


@pytest.mark.parametrize("reflayout", [True, False])
@pytest.mark.parametrize("any_hit", [False, True])
def test_c2_primary_and_bounce(c2, port, reflayout, any_hit):
    from tracer_b200 import harness as H
    prim, scene = c2
    rays = H.cornell_camera_rays(384, 216)
    want = port.trace(prim, rays, any=any_hit, records=True, nthreads=8)
    assert_hits_equal(gpu_trace(scene, rays, any_hit, reflayout), want["hits"], "primary", want["records"])
    bounce, _ = H.bounce_rays(port.trace(prim, rays, records=True, nthreads=8)["records"])
    assert_like_oracle(gpu_trace(scene, bounce, any_hit, reflayout), port, prim, bounce, any_hit, "bounce")


@pytest.mark.parametrize("reflayout", [True, False])
def test_mixed_primitives(refcornell, port, reflayout):
    """Cube + Square + Sphere + Triangle leaves (the reference's actual Cornell leaf mix)."""
    from tracer_b200 import harness as H
    prim, scene = refcornell
    rays = H.cornell_camera_rays(320, 180)
    first = port.trace(prim, rays, records=True, nthreads=8)
    assert_hits_equal(gpu_trace(scene, rays, False, reflayout), first["hits"], "primary", first["records"])
    bounce, _ = H.bounce_rays(first["records"])
    assert_like_oracle(gpu_trace(scene, bounce, False, reflayout), port, prim, bounce, False, "bounce")
    shadow, _ = H.shadow_rays(first["records"], prim.squareList[5:6], prim.squareList[6:7])
    assert_like_oracle(gpu_trace(scene, shadow, True, reflayout), port, prim, shadow, True, "shadow")
    rnd = H.random_rays(100000, seed=5, lo=(-245, 0, 0), hi=(800, 555, 555))
    assert_like_oracle(gpu_trace(scene, rnd, False, reflayout), port, prim, rnd, False, "random")


def test_expand_hits_matches_oracle_records(refcornell, port):
    torch = _torch()
    from tracer_b200 import harness as H, rays_to_torch
    prim, scene = refcornell
    rays = H.cornell_camera_rays(320, 180)
    hits, want = oracle(port, prim, rays)
    d = rays_to_torch(rays, "cuda:0")
    recs = scene.expand(d, scene.hit(d)).cpu().numpy().view(L.record_dtype).reshape(-1)
    assert np.array_equal(recs["hit"], want["hit"])
    m = want["hit"] == 1
    sph = m & (hits["pType"] == L.SPHERE)
    assert sph.sum() > 1000
    for k in ("t", "p", "gn", "sn", "front", "material"):
        assert np.array_equal(recs[k][m].view(np.uint32), want[k][m].view(np.uint32)), k
    assert np.array_equal(recs["uv"][m & ~sph].view(np.uint32), want["uv"][m & ~sph].view(np.uint32))
    assert_sphere_uv(recs["uv"][sph, 0], recs["uv"][sph, 1], want["gn"][sph], want["uv"][sph, 0], want["uv"][sph, 1], "expand")


def test_host_pointer_path_equals_device_path(c2, port):
    from tracer_b200 import harness as H
    prim, scene = c2
    rays = H.random_rays(300000, seed=11, lo=(-245, 0, 0), hi=(800, 555, 555))
    a = gpu_trace(scene, rays, host=False)
    b = gpu_trace(scene, rays, host=True)
    assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    assert_like_oracle(a, port, prim, rays, False, "random")


def test_soup_incoherent(built, port):
    """C5-shaped workload scaled down: 200k-triangle soup, 400k uniform random rays."""
    _torch()
    from tracer_b200 import Scene, harness as H
    prim = H.scene_soup(200000, seed=1, extent=0.01)
    scene = Scene(prim, 0)
    rays = H.random_rays(400000, seed=2)
    want, recs = oracle(port, prim, rays)
    for reflayout in (True, False):
        assert_hits_equal(gpu_trace(scene, rays, False, reflayout), want, f"soup reflayout={reflayout}", recs)
    short = rays.copy(); short["tmax"] = 0.05
    assert_like_oracle(gpu_trace(scene, short, True, False), port, prim, short, True, "soup any, finite tmax")


def test_edge_cases(built, port):
    """Empty batch, single-primitive scene (root is a leaf, SURVEY appendix A note 4), two-leaf scene,
    axis-parallel directions, origin inside boxes, ragged batch sizes around the warp/block size."""
    torch = _torch()
    from tracer_b200 import Scene, harness as H
    tri = H.make_vertices(np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], dtype=np.float32), [[0, 1, 2], [0, 1, 3]])
    one = H.build_primitive(tri, np.array([0, 1, 2], dtype=np.uint32))
    two = H.build_primitive(tri, np.array([0, 1, 2, 0, 1, 3], dtype=np.uint32))
    assert one.bvhList.size == 1 and two.bvhList.size == 3
    for prim in (one, two):
        scene = Scene(prim, 0)
        assert scene.hit(torch.empty((0, 8), dtype=torch.float32, device="cuda:0")).shape[0] == 0
        for n in (1, 31, 32, 33, 255, 257, 1000):
            rays = H.random_rays(n, seed=n, lo=(-0.5, -0.5, -0.5), hi=(1, 1, 1))
            axis = rays.copy()
            axis["d"] = 0; axis["d"][:, n % 3] = 1.0          # axis-parallel: 1/0 = inf slabs
            for r in (rays, axis):
                want, recs = oracle(port, prim, r)
                for reflayout in (True, False):
                    assert_hits_equal(gpu_trace(scene, r, False, reflayout), want, f"n={n}", recs)
        scene.close()
