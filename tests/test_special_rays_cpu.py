"""Special-valued rays and degenerate surfaces: the generators that tests/test_gpu_special_rays.py traces, the proof that each
family of special values actually occurs, and offset_ray on special normals. Nothing here needs a GPU.

trq_ray takes its direction as given and its tmax as Scene::hit's test_t, without restriction, so rays with -0.0, NaN, inf,
denormal or FLT_MAX components, directions that are not unit length and special tmax values all have a defined answer: the
oracle's. offset_ray converts 256 * n to int32 the way x86 does (INT32_MIN for NaN and |256 n| >= 2^31), and adds in the
float's bits modulo 2^32."""
import numpy as np
import pytest

from tracer_b200 import layout as L

from .util import bits

f32 = np.float32
FLT_MIN, FLT_MAX = np.finfo(f32).tiny, np.finfo(f32).max
MAX_DEPTH = 31
# Maximum ulp errors of the single-precision functions, CUDA 12.9 Math API (CUDA C++ Programming Guide, "Mathematical
# Functions", single-precision standard library table; without -use_fast_math)
ULP_ATAN2F, ULP_ASINF, ULP_SINF, ULP_COSF = 3, 2, 2, 2
PI_F, PI_2_F = f32(3.14159265358979323846), f32(1.57079632679489661923)

DIR_FAMILIES = ("plain", "zero1", "zero2", "zero3", "inf", "nan", "denormal", "fltmax", "scaled")
ORIGIN_FAMILIES = ("o_nan", "o_inf", "o_1e30", "o_plane")
FAMILIES = DIR_FAMILIES + ORIGIN_FAMILIES
TMAX_SPECIAL = np.array([np.nan, np.inf, -np.inf, 0.0, -0.0, -1.0, FLT_MIN, np.nextafter(FLT_MIN, f32(1)), 1e-40, FLT_MAX,
                         1e-30, 3.0], dtype=f32)


def _signed(rng, v, n):
    return np.where(rng.random(n) < 0.5, -v, v).astype(f32)


def special_rays(rng, prim, n, n_nan_origin=64):
    """n seeded rays; ray k belongs to FAMILIES[fam[k]] (one special direction or origin), and every fourth ray also has a
    special tmax (TMAX_SPECIAL). NaN-origin rays visit O(nNode) nodes, so at most n_nan_origin of them. -> (rays, fam)"""
    bvh = prim.bvhList
    fin = np.isfinite(bvh["mini"]).all(axis=1) & np.isfinite(bvh["maxi"]).all(axis=1)
    lo, hi = bvh["mini"][fin].min(axis=0), bvh["maxi"][fin].max(axis=0)
    ext = np.maximum(hi - lo, f32(1e-3))
    rays = np.zeros(n, dtype=L.ray_dtype)
    o = rng.uniform(lo - 0.2 * ext, hi + 0.2 * ext, (n, 3)).astype(f32)
    d = rng.normal(size=(n, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(f32)
    fam = rng.integers(0, len(FAMILIES), n)
    fam[:len(FAMILIES)] = np.arange(len(FAMILIES))                       # every family at least once
    nan_o = np.nonzero(fam == FAMILIES.index("o_nan"))[0]
    fam[nan_o[n_nan_origin:]] = 0
    ax = rng.integers(0, 3, n)
    rows = np.arange(n)

    def sel(name):
        return np.nonzero(fam == FAMILIES.index(name))[0]

    k = sel("zero1"); d[k, ax[k]] = _signed(rng, f32(0), k.size)
    k = sel("zero2")
    for j in range(3):
        m = k[ax[k] != j]
        d[m, j] = _signed(rng, f32(0), m.size)
    d[k, ax[k]] = _signed(rng, f32(1), k.size)
    k = sel("zero3"); d[k] = _signed(rng, f32(0), 3 * k.size).reshape(-1, 3)
    k = sel("inf"); d[k, ax[k]] = _signed(rng, f32(np.inf), k.size)
    k = sel("nan"); d[k, ax[k]] = np.nan
    k = sel("denormal")
    den = rng.uniform(1e-45, 1e-38, (k.size, 3)).astype(f32) * _signed(rng, f32(1), 3 * k.size).reshape(-1, 3)
    allden = rng.random(k.size) < 0.3
    d[k[allden]] = den[allden]
    d[k[~allden], ax[k[~allden]]] = den[~allden, 0]
    k = sel("fltmax"); d[k, ax[k]] = _signed(rng, FLT_MAX, k.size)
    k = sel("scaled"); d[k] = d[k] * np.ldexp(f32(1), rng.integers(-100, 101, k.size)).astype(f32)[:, None]
    k = sel("o_nan")
    whole = rng.random(k.size) < 0.5
    o[k[whole]] = np.nan
    o[k[~whole], ax[k[~whole]]] = np.nan
    k = sel("o_inf"); o[k, ax[k]] = _signed(rng, f32(np.inf), k.size)
    k = sel("o_1e30"); o[k, ax[k]] = _signed(rng, f32(1e30), k.size)
    k = sel("o_plane")
    node = bvh[rng.integers(0, bvh.size, k.size)]
    plane = np.where(rng.random(k.size) < 0.5, node["mini"][np.arange(k.size), ax[k]], node["maxi"][np.arange(k.size), ax[k]])
    plane = np.where(plane == 0, f32(-0.0), plane).astype(f32)              # a plane at zero: the origin on it at -0.0
    o[k, ax[k]] = plane
    rays["o"], rays["d"] = o, d
    tm = np.full(n, FLT_MAX, dtype=f32)
    every4 = rows % 4 == 3
    tm[every4] = TMAX_SPECIAL[rng.integers(0, TMAX_SPECIAL.size, every4.sum())]
    tm[:TMAX_SPECIAL.size] = TMAX_SPECIAL                                 # every special tmax at least once
    k = sel("zero3"); tm[k] = np.where(rng.random(k.size) < 0.5, FLT_MIN, f32(1e-30))
    rays["tmax"] = tm
    return rays, fam


def nan_origin_rays(rng, n):
    """Rays whose origin is NaN on every axis: every box test passes, ties go right, so the left child is pushed at every
    level of a tree."""
    rays = np.zeros(n, dtype=L.ray_dtype)
    rays["o"] = np.nan
    d = rng.normal(size=(n, 3))
    rays["d"] = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(f32)
    rays["tmax"] = FLT_MAX
    return rays


def comb_right(depth=MAX_DEPTH):
    """A depth-31 comb whose interior children are all on the right: a ray that enters both children everywhere with a
    tie descends right and pushes every left leaf, so the far-child stack fills to its bound."""
    from .test_gpu_tree_shapes import comb_prim
    prim, topo, lv = comb_prim(depth, interior_left=False)
    return prim


def one_leaf():
    from tracer_b200 import harness as H
    tri = H.make_vertices(np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], dtype=f32), [[0, 1, 2]])
    return H.build_primitive(tri, np.array([0, 1, 2], dtype=np.uint32))


# ------------------------------------------------------------------------------------------------ degenerate surfaces
SPECIAL_NORMALS = np.array([[np.nan, 0, 1], [0, 0, 0], [-0.0, -0.0, -0.0], [-1, -2, -3], [1e8, -1e8, 3], [3e38, -3e38, 3e38],
                            [np.inf, 1, -np.inf], [8388608, -8388607, 0.5], [-2 ** 31 / 256, 2 ** 31 / 256, 1e-40],
                            [np.nextafter(f32(2 ** 23), f32(0)), -2 ** 23, 1]], dtype=f32)


def degenerate_scene():
    """Triangles whose vertex normals are NaN, zero, negative or huge; spheres of radius 0, negative radius, and radius
    1e-12 near (1e3, 1e3, 1e3); cubes with a zero-scale and a NaN model matrix; plus light squares for shadow rays.
    -> (Primitive, targets): one target point per primitive for rays to aim at."""
    from tracer_b200 import harness as H
    ms, targets = H.MeshSoup(), []
    normals = []
    for i, nrm in enumerate(SPECIAL_NORMALS):
        x = f32(3 * i)
        pos = np.array([[x, 0, 0], [x + 2, 0, 0], [x, 2, 0]], dtype=f32)
        ms.add(pos, [[0, 1, 2]])
        normals += [nrm, nrm[::-1], nrm * f32(-1)]
        targets.append(pos.mean(axis=0))
    tri, idx = ms.arrays()
    tri["n"] = np.array(normals, dtype=f32)
    sph = []
    for i, (r, c) in enumerate([(0.0, (2, 10, 0)), (-1.0, (6, 10, 0)), (1e-12, (1000, 1000.5, 1000.25)), (1.5, (0, 20, 0))]):
        s = H.make_sphere(1.0, c, i)
        s["radius"] = f32(r)
        sph.append(s)
        targets.append(np.array(c, dtype=f32))
    cubes = []
    for i in range(2):
        c = H.make_cube(H.translation4x4(10 + 10 * i, -10, 0), i)
        if i == 0:
            c["model"][0] = 0.0                                          # zero scale along x: a flat cube, singular normal matrix
            c["normal"][0] = 0.0
        else:
            c["model"][5] = c["normal"][5] = c["inverse"][5] = np.nan    # a NaN in every matrix of the cube
        cubes.append(c)
        targets.append(np.array([10.0 + 10.5 * i, -9.5, 0.5], dtype=f32))
    squares = [H.make_square(0, (-5, 5), 2, (-5, 5), 1, 30.0, 3), H.make_square(0, (20, 25), 2, (-5, 5), 1, 30.0, 4)]
    prim = H.build_primitive(tri, idx, spheres=np.array(sph, dtype=L.sphere_dtype), cubes=np.array(cubes, dtype=L.cube_dtype),
                             squares=np.array(squares, dtype=L.square_dtype))
    return prim, np.array(targets, dtype=f32)


def aimed_rays(rng, targets, n):
    """Rays from random points around each target, aimed at it (pole rays along y included)."""
    t = targets[rng.integers(0, len(targets), n)]
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    o = (t - 6 * d).astype(f32)
    o[::5] = t[::5] + np.array([0, 6, 0], dtype=f32)
    rays = np.zeros(n, dtype=L.ray_dtype)
    rays["o"] = o
    rays["d"] = (t - o).astype(f32)
    rays["d"][::5] = np.array([0, -1, 0], dtype=f32)
    rays["d"][::10, 0] = -0.0
    from tracer_b200._lib import lib
    lib.trqh_normalize_rays(rays.ctypes.data, n)
    rays["tmax"] = FLT_MAX
    return rays


def pole_spheres_scene():
    """Spheres centred on the axes' zero planes and rays straight along -y / +y with signed-zero x and z: gn.y = +-1 exactly,
    |gn.y| > 1 from rounding, and gn.x, gn.z at +-0 (atan2f / asinf at their special points). -> (Primitive, rays)"""
    from tracer_b200 import harness as H
    rng = np.random.default_rng(77)
    sph, rays = [], []
    for i in range(64):
        r = f32(rng.uniform(0.1, 7)) if i % 2 else f32(i % 8 + 1)
        c = np.array([0.0, 40.0 * i, 0.0], dtype=f32) if i % 4 else np.array([-0.0, 40.0 * i + rng.uniform(0, 1), -0.0], dtype=f32)
        s = H.make_sphere(1.0, c, i)
        s["radius"] = r
        s["box_mini"], s["box_maxi"] = c - abs(r) - 1, c + abs(r) + 1
        sph.append(s)
        for sx in (0.0, -0.0):
            for sz in (0.0, -0.0):
                for dy in (-1.0, 1.0):
                    ray = np.zeros(1, dtype=L.ray_dtype)[0]
                    ray["o"] = (sx, c[1] - dy * f32(rng.uniform(10, 19)), sz)
                    ray["d"] = (np.copysign(0.0, rng.random() - 0.5), dy, np.copysign(0.0, rng.random() - 0.5))
                    ray["tmax"] = FLT_MAX
                    rays.append(ray)
    prim = H.build_primitive(spheres=np.array(sph, dtype=L.sphere_dtype))
    return prim, np.array(rays, dtype=L.ray_dtype)


def flat_cube_scene():
    """Cubes whose local box is flat on one axis at mini = -0.0, maxi = +0.0, with identity-like matrices whose zeros carry
    either sign, and rays starting on that plane: Cube::hit_test ignores range.x, so they are hit at t = 0, and the sign of
    the zero fminf / fmaxf pick reaches uv. -> (Primitive, rays)"""
    from tracer_b200 import harness as H
    rng = np.random.default_rng(31)
    cubes, rays = [], []
    for i in range(24):
        ax = i % 3
        m = np.eye(4, dtype=f32)
        z = m == 0
        m[z] = np.where(rng.random(z.sum()) < 0.5, f32(-0.0), f32(0.0))
        c = np.zeros(1, dtype=L.cube_dtype)[0]
        c["model"] = c["inverse"] = c["normal"] = H.colmajor(m)
        mini, maxi = np.full(3, -1, dtype=f32), np.full(3, 1, dtype=f32)
        mini[ax], maxi[ax] = -0.0, 0.0
        c["box_mini"], c["box_maxi"] = mini, maxi
        c["material"] = i
        cubes.append(c)
    for k in range(4000):
        ax = (k // 8) % 3
        o = rng.uniform(-0.9, 0.9, 3).astype(f32)
        for j in range(3):
            if rng.random() < 0.5:
                o[j] = -0.0 if rng.random() < 0.5 else 0.0
        o[ax] = -0.0 if rng.random() < 0.5 else 0.0
        d = rng.normal(size=3)
        d = (d / np.linalg.norm(d)).astype(f32)
        ray = np.zeros(1, dtype=L.ray_dtype)[0]
        ray["o"], ray["d"], ray["tmax"] = o, d, FLT_MAX
        rays.append(ray)
    prim = H.build_primitive(cubes=np.array(cubes, dtype=L.cube_dtype))
    return prim, np.array(rays, dtype=L.ray_dtype)


# ------------------------------------------------------------------------------------------------ float64 references
def _ulps(x, k):
    """-> (k, ...) array: x stepped -k..k ulps (float32)."""
    out = [x]
    lo = hi = x
    for _ in range(k):
        lo, hi = np.nextafter(lo, f32(-np.inf)), np.nextafter(hi, f32(np.inf))
        out = [lo] + out + [hi]
    return np.stack(out)


def sphere_uv_interval(gn, k_atan2=ULP_ATAN2F, k_asin=ULP_ASINF):
    """Closed interval of sphere uv (Sphere.hh:54-56, intersect.cuh sphere_surface) for shading normals gn: phi and theta
    anywhere within the documented ulp bounds of atan2 / asin, then the float32 chain in the device's order. The chain is
    monotone (u decreasing in phi, v increasing in theta). -> (ulo, uhi, vlo, vhi, u_nearest, v_nearest)"""
    g = gn.astype(np.float64)
    with np.errstate(invalid="ignore"):
        phi = np.arctan2(g[:, 2], g[:, 0]).astype(f32)
        theta = np.arcsin(g[:, 1]).astype(f32)

    def u_of(p):
        return f32(1) - (p + PI_F) / (f32(2) * PI_F)

    def v_of(t):
        return (t + PI_2_F) / PI_F
    p = _ulps(phi, k_atan2)
    t = _ulps(theta, k_asin)
    return u_of(p[-1]), u_of(p[0]), v_of(t[0]), v_of(t[-1]), u_of(phi), v_of(theta)


def _nan_aware_equal(a, b):
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(bits(a)[~na], bits(b)[~nb])


def bounce_direction_candidates(sn, u0, u1):
    """Every direction spawn_bounce can give for shading normal sn and draws (u0, u1) when cosf / sinf return any float32
    within their ulp bounds of cos / sin (float64) at the float32 theta: concentric_sample_disk, z, coordinate_system,
    stw * wi and normalize in float32, in the device's order. -> (m, n_candidates, 3)"""
    with np.errstate(all="ignore"):
        ox, oy = f32(2) * u0 - f32(1), f32(2) * u1 - f32(1)
        xbig = np.abs(ox) > np.abs(oy)
        r = np.where(xbig, ox, oy)
        theta = np.where(xbig, (PI_F / f32(4)) * (oy / ox), PI_F / f32(2) - (PI_F / f32(4)) * (ox / oy)).astype(f32)
        c = _ulps(np.cos(theta.astype(np.float64)).astype(f32), ULP_COSF)
        s = _ulps(np.sin(theta.astype(np.float64)).astype(f32), ULP_SINF)
        cc = np.repeat(c, s.shape[0], axis=0).T                              # (m, nc * ns)
        ss = np.tile(s, (c.shape[0], 1)).T
        origin = (ox == 0) & (oy == 0)
        dx = np.where(origin[:, None], f32(0), r[:, None] * cc)
        dy = np.where(origin[:, None], f32(0), r[:, None] * ss)
        z = np.sqrt(np.fmax(f32(0), (f32(1) - dx * dx) - dy * dy))
        a = sn.astype(f32)
        zero = np.zeros(len(a), dtype=f32)
        b = np.where((np.abs(a[:, 0]) > np.abs(a[:, 1]))[:, None], np.stack([-a[:, 2], zero, a[:, 0]], 1),
                     np.stack([zero, a[:, 2], -a[:, 1]], 1))
        b = b / np.sqrt((b[:, 0] * b[:, 0] + b[:, 1] * b[:, 1]) + b[:, 2] * b[:, 2])[:, None]
        cr = np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1], a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2], a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], 1)
        d = (b[:, None, :] * dx[:, :, None] + cr[:, None, :] * dy[:, :, None]) + a[:, None, :] * z[:, :, None]
        ln = np.sqrt((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2])
        return (d / ln[..., None]).astype(f32)


# ------------------------------------------------------------------------------------------------------------- tests
def test_special_ray_families_occur(built):
    from tracer_b200 import harness as H
    prim = H.scene_reference_cornell()
    rays, fam = special_rays(np.random.default_rng(1), prim, 20000)
    d, o, tm = rays["d"], rays["o"], rays["tmax"]
    assert (fam == FAMILIES.index("o_nan")).sum() == 64
    for name in FAMILIES:
        assert (fam == FAMILIES.index(name)).any(), name
    assert ((d == 0) & np.signbit(d)).any() and ((d == 0) & ~np.signbit(d)).any()
    assert ((d == 0).sum(axis=1) == 3).any() and ((d == 0).sum(axis=1) == 2).any()
    assert (np.isposinf(d).any() and np.isneginf(d).any() and np.isnan(d).any())
    den = (d != 0) & (np.abs(d) < FLT_MIN)
    assert (den & (d > 0)).any() and (den & (d < 0)).any() and (den.sum(axis=1) == 3).any()
    assert (d == FLT_MAX).any() and (d == -FLT_MAX).any()
    with np.errstate(over="ignore", invalid="ignore"):
        ln = np.linalg.norm(d.astype(np.float64), axis=1)
    assert (ln < 2.0 ** -90).any() and (ln > 2.0 ** 90).any()
    assert np.isnan(o).all(axis=1).any() and (np.isnan(o).sum(axis=1) == 1).any()
    assert np.isposinf(o).any() and np.isneginf(o).any() and (o == 1e30).any() and (o == -1e30).any()
    planes = np.concatenate([prim.bvhList["mini"].ravel(), prim.bvhList["maxi"].ravel()])
    on = np.isin(o[fam == FAMILIES.index("o_plane")], planes).any(axis=1)
    assert on.all()
    for v in TMAX_SPECIAL:
        assert (bits(tm) == bits(np.array([v], dtype=f32))[0]).any(), v
    o = special_rays(np.random.default_rng(1), one_leaf(), 2000)[0]["o"]
    assert ((o == 0) & np.signbit(o)).any(), "an origin on a node-box plane at zero, as -0.0"


def test_nan_origin_rays_fill_the_stack_of_the_comb(built, port):
    """On the depth-31 comb with its interior children on the right, a NaN-origin ray descends to the bottom with a pending
    far child at every level: the oracle's stack reaches level 31. The ray ends as a hit on the deepest leaf's right side,
    the first one tested; the oracle defines it."""
    prim = comb_right()
    rays = nan_origin_rays(np.random.default_rng(3), 64)
    out = port.trace(prim, rays, counters=True)
    assert (out["counters"]["max_level"] == MAX_DEPTH).all()
    fam_rays, fam = special_rays(np.random.default_rng(4), prim, 2000)
    out = port.trace(prim, fam_rays, counters=True)
    assert out["counters"]["max_level"][fam == FAMILIES.index("o_nan")].max() == MAX_DEPTH


def _host_offset(p, n):
    from tracer_b200._lib import lib
    p, n = np.ascontiguousarray(p, dtype=f32), np.ascontiguousarray(n, dtype=f32)
    out = np.zeros(3, dtype=f32)
    lib.trqh_offset_ray(p.ctypes.data, n.ctypes.data, out.ctypes.data)
    return out


def _x86_f2i(v):
    v = np.float32(v)
    if np.isnan(v) or v >= 2.0 ** 31 or v < -2.0 ** 31:
        return -2 ** 31
    return int(np.trunc(v))


def _offset_model(p, n):
    """offset_ray in Python integers: of_i = x86 int32(256 n), added into p's bits modulo 2^32."""
    out = np.zeros(3, dtype=f32)
    for k in range(3):
        with np.errstate(over="ignore", invalid="ignore"):
            s = f32(256) * f32(n[k])
        of = _x86_f2i(s) & 0xFFFFFFFF
        pb = int(np.array([p[k]], dtype=f32).view(np.uint32)[0])
        pi = (pb + ((-of) if p[k] < 0 else of)) & 0xFFFFFFFF
        with np.errstate(over="ignore", invalid="ignore"):
            small = f32(p[k]) + f32(1.0 / 65536.0) * f32(n[k])
        out[k] = small if abs(f32(p[k])) < f32(1.0 / 32.0) else np.array([pi], dtype=np.uint32).view(f32)[0]
    return out


def _offset_inputs():
    rng = np.random.default_rng(12)
    ps = [np.array(p, dtype=f32) for p in ([1, -1, 0.01], [-0.0, 0.0, -0.02], [1e3, -1e3, 3e38], [-3e38, 1.5, -2.5],
                                           [np.nan, np.inf, -np.inf], [1e-40, -1e-40, 0.03125])]
    ps += [rng.normal(0, 100, 3).astype(f32) for _ in range(8)]
    ns = list(SPECIAL_NORMALS) + [rng.normal(0, 10.0 ** e, 3).astype(f32) for e in range(-3, 39, 3)]
    return ps, ns


def test_offset_ray_on_special_normals(built, port):
    """trqh_offset_ray (the product's host restatement, whose rule the device follows) equals the oracle's offset_ray and an
    integer model of it on NaN, zero, negative and huge normals: NaN and |256 n| >= 2^31 give of_i = INT32_MIN."""
    ps, ns = _offset_inputs()
    huge = 0
    for p in ps:
        for n in ns:
            host = _host_offset(p, n)
            assert np.array_equal(bits(host), bits(port.offset_ray(p, n))), (p, n)
            assert np.array_equal(bits(host), bits(_offset_model(p, n))), (p, n)
            with np.errstate(over="ignore", invalid="ignore"):
                huge += bool((~(np.abs(f32(256) * n) < 2.0 ** 31)).any())
    assert huge > 0


def test_offset_ray_against_the_reference(reference):
    """The same special normals through the reference's own offset_ray (compiled verbatim on x86)."""
    ps, ns = _offset_inputs()
    for p in ps:
        for n in ns:
            assert np.array_equal(bits(_host_offset(p, n)), bits(reference.offset_ray(p, n))), (p, n)


def test_degenerate_surfaces_reach_the_spawns(built, port):
    """The hits of degenerate_scene carry shading normals with |256 n| >= 2^31 or NaN, from triangles, spheres and cubes;
    the spawns read them."""
    prim, targets = degenerate_scene()
    rays = aimed_rays(np.random.default_rng(2), targets, 6000)
    out = port.trace(prim, rays, records=True)
    rec, hits = out["records"], out["hits"]
    m = rec["hit"] == 1
    with np.errstate(over="ignore", invalid="ignore"):
        big = ~(np.abs(f32(256) * rec["sn"]) < 2.0 ** 31).all(axis=1)
    for kind in (L.TRIANGLE, L.SPHERE):
        assert (m & big & (hits["pType"] == kind)).any(), kind
    assert (m & np.isnan(rec["sn"]).any(axis=1)).any()
    assert (m & (hits["pType"] == L.CUBE)).any()
    assert (m & (hits["pType"] == L.SPHERE) & (hits["pIndex"] == 2)).any(), "the 1e-12 sphere far from the origin"


def test_pole_and_seam_cases_occur(built, port):
    prim, rays = pole_spheres_scene()
    rec = port.trace(prim, rays, records=True)["records"]
    m = rec["hit"] == 1
    gn = rec["gn"][m]
    assert (np.abs(gn[:, 1]) == 1).any() and (np.abs(gn[:, 1]) > 1).any()
    for j in (0, 2):
        z = gn[:, j] == 0
        assert (z & np.signbit(gn[:, j])).any() and (z & ~np.signbit(gn[:, j])).any(), j


def test_flat_cube_hits_at_t_zero(built, port):
    prim, rays = flat_cube_scene()
    out = port.trace(prim, rays, records=True)
    h = out["hits"]
    m = ((h["flags"] & 1) == 1) & (h["pType"] == L.CUBE)
    at0 = m & (h["t"] == 0)
    assert at0.sum() > 50
    uv = np.stack([h["u"], h["v"]], axis=1)[at0]
    assert (uv == 0).any(), "a zero reaches uv"


def test_float64_references_contain_libm(built, port):
    """The float64 references admit what glibc computes: the oracle's sphere uv lies in sphere_uv_interval, and the host
    restatement's bounce directions (glibc cosf / sinf) are among bounce_direction_candidates."""
    from tracer_b200 import harness as H
    prim = H.scene_reference_cornell()
    rays = H.random_rays(200000, seed=3, lo=(-245, 0, 0), hi=(800, 555, 555))
    out = port.trace(prim, rays, records=True, nthreads=8)
    rec, hits = out["records"], out["hits"]
    sph = (rec["hit"] == 1) & (hits["pType"] == L.SPHERE)
    assert sph.sum() > 1000
    ulo, uhi, vlo, vhi, _, _ = sphere_uv_interval(rec["gn"][sph])
    u, v = rec["uv"][sph, 0], rec["uv"][sph, 1]
    assert ((u >= ulo) & (u <= uhi)).all() and ((v >= vlo) & (v <= vhi)).all()
    prim_d, targets = degenerate_scene()
    drec = port.trace(prim_d, aimed_rays(np.random.default_rng(2), targets, 3000), records=True)["records"]
    for recs in (rec[:20000], drec):
        want, src = H.bounce_rays(recs, seed_base=7)
        uu = np.stack([H.pcg32_floats(7 + int(i), 1, 2) for i in src])
        cand = bounce_direction_candidates(recs["sn"][src], uu[:, 0], uu[:, 1])
        d = want["d"]
        same = (bits(cand) == bits(d)[:, None, :]) | (np.isnan(cand) & np.isnan(d)[:, None, :])
        assert same.all(axis=2).any(axis=1).all()
