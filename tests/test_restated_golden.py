"""CPU: the reference comparisons of test_harness, test_oracle_units, test_oracle_golden, test_layout and test_builder, run
against stored answers, so that they also hold where the reference's own build (oracle/_ref) cannot be made.

Those tests feed the workload generators, the oracle's leaf functions and the host BVH builder the inputs below and compare
what comes out with the reference compiled from its source, bit for bit. tests/golden/make_restated_golden.py stores what
the restatements return for exactly those inputs; they are the reference's answers as long as the live comparisons hold,
and `test_stored_answers_are_the_live_references` checks that against the live build wherever it exists. Outputs too large to
store whole are kept as SHA-256 digests."""
import hashlib
import os

import numpy as np
import pytest

from tracer_b200 import harness as H, layout as L
from tracer_b200._lib import lib

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "restated_golden.npz")


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return np.array(h.hexdigest())


def u32(a):
    return np.ascontiguousarray(a).view(np.uint32)


# ------------------------------------------------------------------------------------------------ inputs and answers
def compute_pcg32(port):
    """test_harness.py::test_pcg32_is_the_references"""
    rng = np.random.default_rng(4)
    u, f = [], []
    for _ in range(25):
        seed, seq = int(rng.integers(0, 1 << 62)), int(rng.integers(0, 1 << 62))
        got = np.zeros(64, dtype=np.uint32)
        lib.trqh_pcg32_fill_u32(seed, seq, 64, got.ctypes.data)
        u.append(got)
        f.append(u32(H.pcg32_floats(seed, seq, 64)))
    return {"u": np.stack(u), "f": np.stack(f)}


def compute_camera(port):
    """test_harness.py::test_camera_rays_are_reference_rays / test_camera_rays_are_castray_bit_for_bit"""
    return {"rays_64x36": u32(H.cornell_camera_rays(64, 36)), "rays_32x18": u32(H.cornell_camera_rays(32, 18))}


def compute_spawns(port):
    """test_harness.py: the bounce, shadow and RNG-texture spawn tests, from the primary hits of the 48x27 Cornell frame
    (the oracle's records: bit for bit the reference's, tests/test_oracle_golden.py)."""
    prim = H.scene_reference_cornell()
    la, lb = prim.squareList[5:6], prim.squareList[6:7]
    first = port.trace(prim, H.cornell_camera_rays(48, 27), records=True)["records"]
    out = {"first": digest(first)}
    rays, src = H.bounce_rays(first, seed_base=7)
    out.update(bounce_rays=u32(rays), bounce_src=src)
    rays, src = H.shadow_rays(first, la, lb, seed_base=3)
    out.update(shadow_rays=u32(rays), shadow_src=src)
    n, hit = first.size, first["hit"] == 1
    tex0 = np.random.default_rng(5).integers(0, 1 << 32, size=(n, 4), dtype=np.uint64).astype(np.uint32)
    tex = tex0.copy()
    H.rng_frame_begin(tex)
    rays, _ = H.bounce_rays(first, rng_state=tex)
    out.update(tex_bounce=tex, tex_bounce_rays=u32(rays))
    tex = tex0.copy()
    H.rng_frame_begin(tex)
    sub = np.nonzero(hit)[0].astype(np.uint32)
    rays, _ = H.shadow_rays(first[sub], la, lb, pixel_of=sub, rng_state=tex)
    out.update(tex_shadow=tex, tex_shadow_rays=u32(rays))
    return out


def compute_scene_constants(port):
    """test_harness.py::test_scene_constants_are_the_references"""
    out = {"squares": H.cornell_squares().view(np.uint8), "cubes": H.cornell_cubes().view(np.uint8),
           "spheres": H.cornell_spheres().view(np.uint8)}
    up = np.array((0, 1, 0), dtype=np.float32)
    cams = []
    got = np.zeros(18, dtype=np.float32)
    frm, at = np.array((278, 278, -800), dtype=np.float32), np.array((278, 278, 278), dtype=np.float32)
    lib.trqh_make_camera(frm.ctypes.data, at.ctypes.data, up.ctypes.data, np.float32(45 * (np.pi / 180)),
                         np.float32(1920) / np.float32(1080), np.float32(10.0), got.ctypes.data)
    cams.append(got.copy())
    rng = np.random.default_rng(8)
    for _ in range(20):
        frm, at = rng.uniform(-5, 5, 3).astype(np.float32), rng.uniform(-5, 5, 3).astype(np.float32)
        vfov, aspect, focus = np.float32(rng.uniform(0.3, 1.5)), np.float32(rng.uniform(0.5, 2.5)), np.float32(rng.uniform(1, 20))
        lib.trqh_make_camera(frm.ctypes.data, at.ctypes.data, up.ctypes.data, vfov, aspect, focus, got.ctypes.data)
        cams.append(got.copy())
    out["cameras"] = u32(np.stack(cams))
    return out


def compute_leaf_units(port):
    """test_oracle_units.py: the same random and hand-picked inputs, the oracle's leaf functions' answers."""
    out = {}
    rng = np.random.default_rng(1)
    box = np.zeros(8, dtype=np.float32)
    res = []
    for i in range(3000):
        lo = rng.uniform(-2, 2, 3).astype(np.float32)
        box[0:3], box[4:7] = lo, lo + rng.uniform(0, 2, 3).astype(np.float32)
        o = rng.uniform(-4, 4, 3).astype(np.float32)
        d = rng.normal(size=3).astype(np.float32)
        if i % 5 == 0:
            d[rng.integers(3)] = 0.0
        if i % 7 == 0:
            o = (box[0:3] + box[4:7]) / 2
        if i % 11 == 0:
            o[0] = box[0]
        d = (d / np.linalg.norm(d)).astype(np.float32)
        r = np.array([L.FLT_MIN, rng.uniform(0.01, 10)], dtype=np.float32)
        h, t = port.aabb_hit_t(box, o, d, r)
        res.append((int(h), int(np.float32(t if h else 0).view(np.uint32)), int(port.aabb_hit(box, o, d, r))))
    out["aabb"] = np.array(res, dtype=np.uint32)

    rng = np.random.default_rng(2)
    res, recs = [], []
    for i in range(2000):
        pos = rng.uniform(-1, 1, (3, 3)).astype(np.float32)
        if i % 50 == 0:
            pos[2] = pos[0] + (pos[1] - pos[0]) * np.float32(0.5)
        tv = H.make_vertices(pos, [[0, 1, 2]])
        tv["n"] = rng.normal(size=(3, 3)).astype(np.float32)
        tv["uv"] = rng.uniform(0, 1, (3, 2)).astype(np.float32)
        o = rng.uniform(-3, 3, 3).astype(np.float32)
        target = pos.mean(0) if i % 3 else pos[i % 3]
        d = (target - o); d = (d / np.linalg.norm(d)).astype(np.float32)
        r = np.array([L.FLT_MIN, L.FLT_MAX], dtype=np.float32)
        h, rr, rec, _ = port.triangle_hit(tv, [0, 1, 2], o, d, r)
        tie = below = 0
        if h:
            tie = int(port.triangle_hit(tv, [0, 1, 2], o, d, np.array([L.FLT_MIN, rec["t"]], dtype=np.float32))[0])
            below = int(port.triangle_hit(tv, [0, 1, 2], o, d, np.array([L.FLT_MIN, np.nextafter(rec["t"], np.float32(0))],
                                                                           dtype=np.float32))[0])
        res.append((int(h), *u32(rr), tie, below))
        recs.append(rec if h else np.zeros((), dtype=L.record_dtype))
    out["triangle"], out["triangle_records"] = np.array(res, dtype=np.uint32), digest(np.array(recs, dtype=L.record_dtype))

    rng = np.random.default_rng(3)
    spheres, squares, cubes = H.cornell_spheres(), H.cornell_squares(), H.cornell_cubes()
    res, recs = [], []
    for i in range(3000):
        o = rng.uniform((-245, 0, 0), (800, 555, 555)).astype(np.float32)
        d = rng.normal(size=3).astype(np.float32); d = (d / np.linalg.norm(d)).astype(np.float32)
        r = np.array([L.FLT_MIN, L.FLT_MAX if i % 2 else rng.uniform(1, 900)], dtype=np.float32)
        s = spheres[i % len(spheres)]
        if i % 9 == 0:
            o = s["center"] + rng.uniform(-10, 10, 3).astype(np.float32)
        row = []
        for fn, obj in ((port.sphere_hit, s), (port.square_hit, squares[i % len(squares)]), (None, cubes[i % len(cubes)])):
            if fn is None:
                if i % 4 == 0:
                    m = np.asarray(obj["model"]).reshape(4, 4).T
                    o = (m @ np.append(rng.uniform(0.1, 0.9, 3), 1.0).astype(np.float32))[:3].astype(np.float32)
                fn = port.cube_hit
            h, rr, rec = fn(obj, o, d, r)
            row += [int(h), *u32(rr)]
            recs.append(rec if h else np.zeros((), dtype=L.record_dtype))
        res.append(row)
    out["sphere_square_cube"] = np.array(res, dtype=np.uint32)
    out["sphere_square_cube_records"] = digest(np.array(recs, dtype=L.record_dtype))

    q = H.cornell_squares()[2]
    o, d = np.array([100, 555, 100], dtype=np.float32), np.array([1, 0, 0], dtype=np.float32)
    r = np.array([L.FLT_MIN, L.FLT_MAX], dtype=np.float32)
    parallel = [port.square_hit(q, o, d, r)[0]]
    o[1] = 500
    parallel.append(port.square_hit(q, o, d, r)[0])
    out["square_parallel"] = np.array(parallel, dtype=np.uint32)

    rng = np.random.default_rng(4)
    res = []
    for i in range(2000):
        p = rng.uniform(-600, 600, 3).astype(np.float32)
        if i % 3 == 0:
            p *= np.float32(1e-3)
        if i % 17 == 0:
            p[0] = 0.0
        n = rng.normal(size=3).astype(np.float32); n = (n / np.linalg.norm(n)).astype(np.float32)
        host = np.zeros(3, dtype=np.float32)
        lib.trqh_offset_ray(p.ctypes.data, n.ctypes.data, host.ctypes.data)
        ray = np.zeros(1, dtype=L.ray_dtype); ray["d"][0] = rng.uniform(-5, 5, 3)
        lib.trqh_normalize_rays(ray.ctypes.data, 1)
        res.append(np.concatenate([u32(port.offset_ray(p, n)), u32(host), u32(ray["d"][0])]))
    out["offset_ray_ctor"] = np.stack(res)
    return out


def compute_random_scenes(port):
    """test_oracle_golden.py::test_port_vs_reference_random_scenes: the oracle's records, as digests."""
    prim = H.scene_reference_cornell()
    rays = H.cornell_camera_rays(160, 90)
    first = port.trace(prim, rays, records=True, nthreads=4)["records"]
    out = {}
    for k, (r, any_hit) in enumerate(((rays, False), (H.bounce_rays(first)[0], False),
                                      (H.shadow_rays(first, prim.squareList[5:6], prim.squareList[6:7])[0], True),
                                      (H.random_rays(20000, seed=5, lo=(-245, 0, 0), hi=(800, 555, 555)), False))):
        out[f"cornell{k}"] = digest(port.trace(prim, r, any=any_hit, records=True, nthreads=4)["records"])
    soup = H.scene_soup(20000, seed=8, extent=0.05)
    out["soup"] = digest(port.trace(soup, H.random_rays(20000, seed=6), records=True, nthreads=4)["records"])
    return out


def _tree(leaves):
    import ctypes as C
    n = leaves.size
    nodes = np.zeros(2 * n - 1, dtype=L.bvh_dtype)
    nodes[:n] = leaves
    nn, md = C.c_uint32(0), C.c_uint32(0)
    assert lib.trq_bvh_build_tree(nodes.ctypes.data, n, C.byref(nn), C.byref(md)) == 0
    return nodes


def _leaves(prim):
    n = int((prim.bvhList["pType"] != L.BVH).sum())
    leaves = prim.bvhList[1:n + 1].copy()
    leaves["parent"] = 0
    return leaves


def compute_builder(port):
    """test_builder.py::test_tree_equals_reference_builder_live / test_c3_tree_equals_reference_builder: the host builder's
    trees (padding words zeroed, as the reference leaves them undefined), as digests."""
    prims = [H.scene_soup(n, seed=100 + n, extent=e) for n, e in ((20000, 0.02), (5000, 0.3), (333, 1.0))]
    prims += [H.scene_reference_cornell(), H.scene_c2(), H.scene_c1()]
    out = {}
    for k, prim in enumerate(prims):
        tree = _tree(_leaves(prim))
        tree["pad"] = 0
        out[f"scene{k}"] = digest(tree)
    rng = np.random.default_rng(123)
    lattice = []
    for _ in range(40):
        n = int(rng.integers(2, 40))
        lv = np.zeros(n, dtype=L.bvh_dtype)
        lo = rng.integers(-2, 3, (n, 3)).astype(np.float32)
        lv["mini"], lv["maxi"] = lo, lo + rng.integers(0, 3, (n, 3)).astype(np.float32)
        lv["pType"], lv["pIndex"] = L.TRIANGLE, np.arange(n)
        lattice.append(_tree(lv))
    out["lattice"] = digest(*lattice)
    c3 = H.scene_c3(2).bvhList.copy()
    c3["pad"] = 0
    out["c3"] = digest(c3)
    return out


COMPUTE = {"pcg32": compute_pcg32, "camera": compute_camera, "spawns": compute_spawns, "constants": compute_scene_constants,
           "leaf": compute_leaf_units, "scenes": compute_random_scenes, "builder": compute_builder}


# ------------------------------------------------------------------------------------------------ the checks
@pytest.fixture(scope="module")
def stored():
    return np.load(GOLDEN)


@pytest.mark.parametrize("group", sorted(COMPUTE))
def test_restatements_give_the_stored_reference_answers(built, port, stored, group):
    got = COMPUTE[group](port)
    want = sorted(k.split("/", 1)[1] for k in stored.files if k.startswith(group + "/"))
    assert sorted(got) == want
    for k, v in got.items():
        w = stored[f"{group}/{k}"]
        assert v.shape == w.shape and np.array_equal(v, w), \
            f"{group}/{k} differs" + ("" if v.dtype.kind == "U" else f" at {np.argwhere(v != w)[:5].tolist()}")


def test_rng_texel_entry_and_exit_known_answer(built):
    """toRNG fills pcg32_t {state, inc} positionally with (inc, state) (Render.hh:96-120): a texel that draws nothing in a
    frame comes out with its halves traded."""
    tex = np.array([[0x11111111, 0x22222222, 0x33333333, 0x44444444]], dtype=np.uint32)
    H.rng_frame_begin(tex)
    rays, _ = H.bounce_rays(np.zeros(1, dtype=L.record_dtype), rng_state=tex)
    assert rays.size == 0 and tex[0].tolist() == [0x33333333, 0x44444444, 0x11111111, 0x22222222]


def test_layout_offsets_of_the_reference_headers():
    """sizeof / offsetof of the reference's structs (test_layout.py::test_against_reference_headers) as that test found them."""
    off = lambda dt, f: dt.fields[f][1]
    assert (off(L.bvh_dtype, "pType"), off(L.bvh_dtype, "pIndex"), off(L.bvh_dtype, "mini")) == (16, 20, 32)
    assert (off(L.sphere_dtype, "center"), off(L.sphere_dtype, "material"), off(L.sphere_dtype, "box_mini")) == (16, 224, 240)
    assert (off(L.square_dtype, "range_i"), off(L.square_dtype, "range_j"), off(L.square_dtype, "axis_k"),
            off(L.square_dtype, "value_k")) == (8, 16, 24, 28)
    assert (off(L.square_dtype, "model"), off(L.square_dtype, "material"), off(L.square_dtype, "box_mini")) == (32, 224, 240)
    assert (off(L.cube_dtype, "inverse"), off(L.cube_dtype, "box_mini"), off(L.cube_dtype, "material")) == (128, 192, 224)


def test_stored_answers_are_the_live_references(port, reference, reference_setup, reference_builder, stored):
    """Where the reference's own build exists: the stored answers are still what it returns (spot checks of every group)."""
    rng = np.random.default_rng(4)
    for i in range(25):
        seed, seq = int(rng.integers(0, 1 << 62)), int(rng.integers(0, 1 << 62))
        u, f = reference.pcg32(seed, seq, 64)
        assert np.array_equal(u, stored["pcg32/u"][i]) and np.array_equal(u32(f), stored["pcg32/f"][i])
    prim = H.scene_reference_cornell()
    first = reference.trace(prim, H.cornell_camera_rays(48, 27))
    assert np.array_equal(u32(H.bounce_rays(first, seed_base=7)[0]), stored["spawns/bounce_rays"])
    assert np.array_equal(u32(reference_setup.prepare_camera(1920, 1080)), stored["constants/cameras"][0])
    for k, prim in enumerate([H.scene_reference_cornell(), H.scene_c2(), H.scene_c1()]):
        assert digest(reference_builder.build_tree(_leaves(prim))) == stored[f"builder/scene{k + 3}"]
