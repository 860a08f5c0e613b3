"""The device-resident wavefront (cast -> trace -> spawn -> trace_indirect ...): the cameras, sizes and seed bases that
tests/test_gpu_wavefront.py runs, the comparison rules it applies, and the proof that those rules are sharp and that every
case family actually occurs. Nothing here needs a GPU.

Rules: camera, bounce and shadow rays against the host restatements (tracer_b200/harness.py, pinned to the reference by
tests/test_harness.py) byte for byte, NaN-aware; bounce directions by test_gpu_special_rays.assert_bounce_directions where
the device's bits differ from the host's (glibc cosf / sinf); shadow lengths (strict fp32 sqrtf on both sides) bit for bit;
sphere uv by assert_sphere_uv."""
import math

import numpy as np
import pytest

from tracer_b200 import layout as L

from .test_special_rays_cpu import _nan_aware_equal, assert_sphere_uv, sphere_uv_interval
from .util import bits

f32 = np.float32
PI_F = f32(math.pi)

# the bench's cameras (bench.py: c2 / c3path cast the Cornell camera, c1 traces RT_Nextweek's camera0)
CORNELL_CAMERA = ((278, 278, -800), (278, 278, 278), (0, 1, 0), f32(45 * (math.pi / 180)), 10.0)
C1_CAMERA = ((13, 2, 3), (0, 0, 0), (0, 1, 0), f32(20 * math.pi / 180), 10.0)
BENCH_CASTS = (("cornell 1920x1080", CORNELL_CAMERA, 1920, 1080), ("cornell 3840x2160", CORNELL_CAMERA, 3840, 2160),
               ("c1 1280x720", C1_CAMERA, 1280, 720))
# 1x1, one column, one row, W*H not a multiple of the 256-thread block, and both sides odd around 256
CAST_SIZES = ((1, 1), (1, 77), (300, 1), (4097, 3), (255, 257))
# the bench's per-rank seed bases (rank << 32) and one whose seedBase + i wraps past 2^64
SEED_BASES = tuple(r << 32 for r in range(8)) + ((1 << 64) - 1000,)


def random_cameras(rng, n=50):
    """n seeded cameras (lookFrom, lookAt, viewUp, vfov in (0, pi), focus_dist), float32 values, with a W x H each."""
    out = []
    for _ in range(n):
        frm = rng.uniform(-500, 500, 3).astype(f32)
        d = rng.normal(size=3)
        at = (frm + d / np.linalg.norm(d) * rng.uniform(0.01, 1000)).astype(f32)
        up = rng.normal(size=3).astype(f32)
        vfov = f32(rng.uniform(1e-3, math.pi - 1e-3))
        focus = f32(rng.uniform(0.05, 100))
        out.append(((tuple(frm), tuple(at), tuple(up), vfov, focus), int(rng.integers(1, 200)), int(rng.integers(1, 200))))
    return out


def degenerate_cameras():
    """-> [(family, camera)]: cameras the reference's MakeCamera accepts but that give NaN / inf / degenerate rays."""
    frm, at, up, vfov, focus = (3.0, 2.0, 1.0), (0.0, 0.5, 0.0), (0.0, 1.0, 0.0), f32(0.7), f32(4.0)
    return [("lookAt = lookFrom", (frm, frm, up, vfov, focus)),
            ("viewUp parallel to the view", ((0.0, 5.0, 0.0), (0.0, 0.0, 0.0), (0.0, 2.0, 0.0), vfov, focus)),
            ("viewUp zero", (frm, at, (0.0, 0.0, 0.0), vfov, focus)),
            ("vfov 0", (frm, at, up, f32(0), focus)),
            ("vfov pi", (frm, at, up, PI_F, focus)),
            ("focus_dist 0", (frm, at, up, vfov, f32(0))),
            ("focus_dist negative", (frm, at, up, vfov, f32(-3.5)))]


def host_camera_rays(cam, W, H):
    from tracer_b200 import harness as H_
    frm, at, up, vfov, focus = cam
    return H_.camera_rays(frm, at, vfov, W, H, up=up, focus=focus)


def assert_rays_equal(got, want, where):
    """trq_ray arrays NaN-aware bit for bit (a NaN made by float arithmetic has no agreed payload)."""
    assert got.size == want.size, f"{where}: {got.size} rays, want {want.size}"
    for k in ("o", "d", "tmax"):
        assert _nan_aware_equal(np.ascontiguousarray(got[k]).reshape(-1), np.ascontiguousarray(want[k]).reshape(-1)), \
            f"{where}: ray {k} differs"


def assert_shadow_lengths(got, want, where):
    """Shadow tmax = sqrtf(dot(dirv, dirv)) in strict fp32 on the device and the host: bit for bit."""
    bad = np.nonzero(bits(got) != bits(want))[0]
    assert bad.size == 0, f"{where}: {bad.size} shadow lengths differ, first {bad[:3]}: {got[bad[:3]]} want {want[bad[:3]]}"


def pcg32_first_two(seeds):
    """The two draws spawn_bounce takes from PCG32(seed, 1) (pcg_basic.c:44-67), for an array of uint64 seeds at once."""
    mul, inc = np.uint64(6364136223846793005), np.uint64(3)           # inc = (1 << 1) | 1
    state = np.asarray(seeds, dtype=np.uint64) + inc                   # srandom: next() from 0, += seed, next()
    state = state * mul + inc
    out = []
    for _ in range(2):
        old = state
        state = old * mul + inc
        x = (((old >> np.uint64(18)) ^ old) >> np.uint64(27)).astype(np.uint32)
        rot = (old >> np.uint64(59)).astype(np.uint32)
        r = (x >> rot) | (x << ((np.uint32(32) - rot) & np.uint32(31)))
        out.append(r.astype(f32) * f32(2.0 ** -32))
    return np.stack(out, axis=1)


def subsample(n, ptype, stride=16):
    """Rays checked against the oracle at full size: every `stride`-th, plus every sphere / cube / square hit."""
    return np.unique(np.concatenate([np.arange(0, n, stride), np.nonzero(ptype[:n] != L.TRIANGLE)[0]]))


# ------------------------------------------------------------------------------------------------------------- tests
def _sphere_hits(port):
    from tracer_b200 import harness as H
    prim = H.scene_c1()
    rays = host_camera_rays(C1_CAMERA, 320, 180)
    out = port.trace(prim, rays, records=True, nthreads=8)
    h, r = out["hits"], out["records"]
    m = (r["hit"] == 1) & (h["pType"] == L.SPHERE)
    gn = r["gn"][m]
    with np.errstate(invalid="ignore"):
        plain = np.isfinite(gn).all(axis=1) & (gn[:, 0] != 0) & (gn[:, 2] != 0) & (np.abs(gn[:, 1]) < 1)
    return r["uv"][m][plain], gn[plain]


def test_sphere_uv_rule_rejects_one_ulp_past_the_bound(built, port):
    """The interval's edges pass; a u or v one ulp past either edge fails, at every sphere hit tried."""
    uv, gn = _sphere_hits(port)
    assert gn.shape[0] > 5000
    ulo, uhi, vlo, vhi, unear, vnear = sphere_uv_interval(gn)
    assert_sphere_uv(unear, vnear, gn, unear, vnear, "nearest")
    assert_sphere_uv(ulo, vhi, gn, unear, vnear, "edges")
    assert_sphere_uv(uhi, vlo, gn, unear, vnear, "edges")
    for k in range(0, gn.shape[0], 997):
        g = gn[k:k + 1]
        for name, u, v in (("u below", np.nextafter(ulo[k:k + 1], f32(-np.inf)), vnear[k:k + 1]),
                           ("u above", np.nextafter(uhi[k:k + 1], f32(np.inf)), vnear[k:k + 1]),
                           ("v below", unear[k:k + 1], np.nextafter(vlo[k:k + 1], f32(-np.inf))),
                           ("v above", unear[k:k + 1], np.nextafter(vhi[k:k + 1], f32(np.inf)))):
            with pytest.raises(AssertionError, match="outside"):
                assert_sphere_uv(u, v, g, unear[k:k + 1], vnear[k:k + 1], name)


def test_shadow_length_rule_rejects_one_ulp(built, port):
    from tracer_b200 import harness as H
    prim = H.scene_reference_cornell()
    recs = port.trace(prim, host_camera_rays(CORNELL_CAMERA, 64, 36), records=True, nthreads=8)["records"]
    sh, _ = H.shadow_rays(recs, prim.squareList[5:6], prim.squareList[6:7], seed_base=3)
    assert sh.size > 1000
    assert_shadow_lengths(sh["tmax"], sh["tmax"].copy(), "same")
    for k in (0, sh.size // 2, sh.size - 1):
        for step in (np.inf, -np.inf):
            t = sh["tmax"].copy()
            t[k] = np.nextafter(t[k], f32(step))
            with pytest.raises(AssertionError, match="shadow lengths differ"):
                assert_shadow_lengths(t, sh["tmax"], "1 ulp")
    off = sh.copy()
    off["d"][7, 1] = np.nextafter(off["d"][7, 1], f32(np.inf))
    with pytest.raises(AssertionError, match="ray d differs"):
        assert_rays_equal(off, sh, "1 ulp")


def test_camera_families_occur(built):
    """Each degenerate camera gives the pattern it stands for on the host; random and bench cameras give finite unit rays."""
    seen = {}
    for family, cam in degenerate_cameras():
        r = host_camera_rays(cam, 33, 17)
        d = r["d"]
        nan, fin = np.isnan(d).any(axis=1), np.isfinite(d).all(axis=1)
        same = (bits(d) == bits(d[:1])).all()
        seen[family] = (bool(nan.all()), bool(fin.all()), bool(same))
    assert seen["lookAt = lookFrom"][0] and seen["viewUp parallel to the view"][0] and seen["viewUp zero"][0]
    assert seen["focus_dist 0"][0]                                 # sample == origin: normalize(0)
    assert seen["vfov 0"][1] and seen["vfov 0"][2]                 # every ray along -w
    assert seen["vfov pi"][1] and not seen["vfov pi"][2]           # tanf(pi_f / 2) is a huge finite value
    assert seen["focus_dist negative"][1]
    neg = host_camera_rays(degenerate_cameras()[-1][1], 33, 17)
    pos = host_camera_rays(degenerate_cameras()[-1][1][:4] + (f32(3.5),), 33, 17)
    assert ((neg["d"] * pos["d"]).sum(axis=1) < -0.999).all()       # every term of sample - origin changes sign
    for cam, W, H in random_cameras(np.random.default_rng(1)):
        r = host_camera_rays(cam, W, H)
        assert r.size == W * H and np.isfinite(r["d"]).all()
    assert {(W * H) % 256 != 0 for W, H in CAST_SIZES} == {True} and any(W == 1 for W, _ in CAST_SIZES) and any(H == 1 for _, H in CAST_SIZES)


def test_seed_base_cases_occur(built):
    """The bench's bases r << 32 select different PCG32 streams (the high word matters), and 2^64 - 1000 + i wraps for
    i >= 1000: the host draws of ray i equal those of base 0 at ray i - 1000."""
    from tracer_b200 import harness as H
    draws = {tuple(H.pcg32_floats(b, 1, 2)) for b in SEED_BASES[:8]}
    assert len(draws) == 8
    seeds = [b + i for b in SEED_BASES[:8] for i in (0, 1, 77777)] + [(SEED_BASES[-1] + i) % (1 << 64) for i in range(0, 3000, 7)]
    assert np.array_equal(pcg32_first_two(seeds), np.stack([H.pcg32_floats(x, 1, 2) for x in seeds]))
    wrap = SEED_BASES[-1]
    for i in (1000, 1001, 123456):
        assert np.array_equal(H.pcg32_floats((wrap + i) % (1 << 64), 1, 2), H.pcg32_floats(i - 1000, 1, 2))
    assert not np.array_equal(H.pcg32_floats(wrap + 999, 1, 2), H.pcg32_floats(0, 1, 2))
    prim = H.scene_reference_cornell()
    from oracle.pyoracle import Port
    recs = Port().trace(prim, host_camera_rays(CORNELL_CAMERA, 64, 36), records=True, nthreads=8)["records"]
    a, sa = H.bounce_rays(recs, seed_base=wrap)
    b, sb = H.bounce_rays(recs, seed_base=0)
    assert np.array_equal(sa, sb) and sa.max() >= 1000               # the wrapped seeds are used
    assert not np.array_equal(bits(a["d"]), bits(b["d"]))
