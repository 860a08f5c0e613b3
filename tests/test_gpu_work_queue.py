"""GPU: the layer between a caller's batch and the per-ray walk -- launch_trace and the persistent work queue of
trace_packed_kernel -- gives the same bytes whatever it is asked to do.

  * A launch captured into a CUDA graph owns its work-queue head: two graphs captured 4096 launches apart (which shared a
    head of the eager ring of 4096 before) replay concurrently on two streams, and each alone, with the eager results.
  * Every scheduler setting (TRQ_REFILL_MIN, TRQ_LEAF_BATCH, TRQ_BLOCKS_PER_SM, TRQ_SORT_RAYS, the compile-time
    TRQ_INTERIOR_UNROLL / TRQ_WAIT_MUL) gives the default's bytes, in both launch configurations, both hit modes and both
    record formats, on the three leaf-specialised kernels and a depth-31 tree. These knobs are read once per process, so
    each setting runs in a worker process: `python -m tests.test_gpu_work_queue worker <in.npz> <out.npz>`.
  * Staged top-of-tree prefixes of every size (TRQ_TOP_NODES) equal the oracle.
  * Batches past the per-launch limit are split into launches that land every record at its own index: a variant built
    with a 2^16-ray limit, and 2^31 + 4097 rays through the product library where the GPU has the memory.
"""
import json
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from tracer_b200 import layout as L

from .test_gpu_fuzz import adversarial_rays
from .test_gpu_parity import _torch, assert_hits_equal, assert_like_oracle, gpu_trace, oracle
from .test_gpu_tree_shapes import MAX_DEPTH, comb_prim, comb_rays

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32
KNOBS = ("TRQ_REFILL_MIN", "TRQ_LEAF_BATCH", "TRQ_BLOCKS_PER_SM", "TRQ_SORT_RAYS", "TRQ_CFG", "TRQ_TOP_NODES", "TRQ_AUTO_SORT",
         "TRQ_NO_SORT", "TRQ_LIB")
PRIM_FIELDS = ("sphereList", "squareList", "cubeList", "triList", "idxList", "bvhList")
SETTINGS = {                                             # one knob moved at a time from the defaults (20 / 12 / fit / flag)
    "refill1": {"TRQ_REFILL_MIN": "1"}, "refill2": {"TRQ_REFILL_MIN": "2"},
    "refill31": {"TRQ_REFILL_MIN": "31"}, "refill32": {"TRQ_REFILL_MIN": "32"},
    "leaf1": {"TRQ_LEAF_BATCH": "1"}, "leaf32": {"TRQ_LEAF_BATCH": "32"},
    "blocks1": {"TRQ_BLOCKS_PER_SM": "1"}, "sort": {"TRQ_SORT_RAYS": "1"},
    "refill1_leaf1": {"TRQ_REFILL_MIN": "1", "TRQ_LEAF_BATCH": "1"},
    "refill32_leaf32": {"TRQ_REFILL_MIN": "32", "TRQ_LEAF_BATCH": "32"},
}
VARIANTS = {                                             # compile-time scheduler constants (trace_kernels.cuh), and the split
    "unroll1": ["-DTRQ_INTERIOR_UNROLL=1"], "unroll3": ["-DTRQ_INTERIOR_UNROLL=3"], "unroll4": ["-DTRQ_INTERIOR_UNROLL=4"],
    "wait0": ["-DTRQ_WAIT_MUL=0"], "wait8": ["-DTRQ_WAIT_MUL=8"],
    "maxrays16": ["-DTRQ_MAX_RAYS_PER_LAUNCH=65536ull"],
}


def _unit(v):
    v = np.asarray(v, dtype=f32)
    return (v / np.linalg.norm(v, axis=-1, keepdims=True)).astype(f32)


def _nan_rays(n):
    """Rays with an all-NaN origin: they enter every box (trq_ray) and walk the whole tree."""
    r = np.zeros(n, dtype=L.ray_dtype)
    r["o"] = np.nan
    r["d"] = _unit([0.3, 0.5, 0.8])
    r["tmax"] = L.FLT_MAX
    return r


def _soup():
    from tracer_b200 import harness as H
    return H.scene_soup(200000, seed=1, extent=0.01)


@pytest.fixture(scope="module")
def soup(built):
    _torch()
    return _soup()


# ---------------------------------------------------------------------------------------------------------------- heads
def test_graphs_captured_4096_launches_apart_replay_concurrently(soup, port):
    """G1 (about 1 M rays ending in 32 all-NaN-origin rays: one warp walks the whole 200 K-triangle tree long after the
    rest of the batch is done) and G2 (another 1 M rays) are captured with exactly 4095 packed-kernel launches between
    them. Replayed on two streams without synchronisation, and then each alone, both give the eager results of a second
    Scene object, which are checked against the oracle on a subsample."""
    torch = _torch()
    from tracer_b200 import Scene, harness as H, rays_to_torch
    prim = soup
    n = 1 << 20
    A = np.concatenate([H.random_rays(n, seed=31), _nan_rays(32)])
    B = H.random_rays(n, seed=32)
    dA, dB = rays_to_torch(A, "cuda:0"), rays_to_torch(B, "cuda:0")
    ref = Scene(prim, 0)
    wantA, wantB = ref.hit(dA, sort=False).clone(), ref.hit(dB, sort=False).clone()
    torch.cuda.synchronize()
    ref.close()
    for rays, want, where in ((A, wantA, "A"), (B, wantB, "B")):
        sub = np.unique(np.concatenate([np.arange(0, rays.size, 997), np.arange(rays.size - 40, rays.size)]))
        got = want.cpu().numpy().view(L.hit_dtype).reshape(-1)[sub]
        assert_like_oracle(got, port, prim, np.ascontiguousarray(rays[sub]), False, f"eager {where}")

    scene = Scene(prim, 0)
    outA, outB = torch.empty_like(wantA), torch.empty_like(wantB)
    one = dB[:1].clone()
    one_out = torch.empty((1, 8), dtype=torch.float32, device="cuda:0")
    side = torch.cuda.Stream()
    g1, g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    with torch.cuda.graph(g1, stream=side):
        scene.hit(dA, sort=False, out=outA)
    for _ in range(4095):                                      # launch k + 1 .. k + 4095 (G1 was launch k)
        scene.hit(one, sort=False, out=one_out)
    with torch.cuda.graph(g2, stream=side):
        scene.hit(dB, sort=False, out=outB)                    # launch k + 4096
    torch.cuda.synchronize()

    X, Y = torch.cuda.Stream(), torch.cuda.Stream()

    def check(what):
        assert torch.equal(outA.view(torch.int32), wantA.view(torch.int32)), \
            f"{what}: G1 differs on {int((outA.view(torch.int32) != wantA.view(torch.int32)).any(dim=1).sum())} rays"
        assert torch.equal(outB.view(torch.int32), wantB.view(torch.int32)), \
            f"{what}: G2 differs on {int((outB.view(torch.int32) != wantB.view(torch.int32)).any(dim=1).sum())} rays"

    def poison():
        outA.view(torch.int32).fill_(-1)                       # flags 0xFFFFFFFF: no record (a miss is all zeros)
        outB.view(torch.int32).fill_(-1)
        X.wait_stream(torch.cuda.current_stream())
        Y.wait_stream(torch.cuda.current_stream())

    poison()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(X):
        t0.record()
        g1.replay()
        t1.record()
    with torch.cuda.stream(Y):
        g2.replay()
    torch.cuda.synchronize()
    print(f"G1 replay {t0.elapsed_time(t1):.1f} ms (G2 replayed beside it)")
    check("concurrent replays")
    poison()
    with torch.cuda.stream(X):
        g1.replay()
    torch.cuda.synchronize()
    with torch.cuda.stream(Y):
        g2.replay()
    torch.cuda.synchronize()
    check("replays one after the other")
    del g1, g2
    scene.close()


# ---------------------------------------------------------------------------------------------- every scheduler setting
def _away_rays(rng, lo, hi, n):
    """Rays that start outside the root box and point away from it: root-box misses."""
    c, r = (lo + hi) * f32(0.5), f32(np.linalg.norm(hi - lo))
    u = _unit(rng.normal(size=(n, 3)))
    rays = np.zeros(n, dtype=L.ray_dtype)
    rays["o"] = (c + f32(2) * r * u).astype(f32)
    rays["d"] = u
    rays["tmax"] = L.FLT_MAX
    return rays


def _ray_sets(name, prim, lv=None):
    """-> [(set name, rays, count or None)]: count = the device-resident batch size of trq_trace_indirect."""
    from tracer_b200 import harness as H
    rng = np.random.default_rng(sum(map(ord, name)))
    seed = lambda: int(rng.integers(1 << 30))
    lo, hi = prim.bvhList["mini"][0].astype(f32), prim.bvhList["maxi"][0].astype(f32)
    pad, c, diag = f32(0.2) * (hi - lo), (lo + hi) * f32(0.5), f32(np.linalg.norm(hi - lo))
    sets = [("adversarial", adversarial_rays(rng, prim, 6000), None),
            ("random", H.random_rays(70000, seed=seed(), lo=lo - pad, hi=hi + pad), None)]   # >= 65536: TRQ_SORT_RAYS orders it
    if name == "c1":
        sets.append(("camera", H.camera_rays((13, 2, 3), (0, 0, 0), f32(20 * np.pi / 180), 96, 64), None))
    else:
        sets.append(("camera", H.camera_rays(c + np.array([0.3, 0.5, -2.5], dtype=f32) * diag, c, f32(0.8), 96, 64), None))
    for n in (1, 31, 33, 4097):
        sets.append((f"n{n}", H.random_rays(n, seed=seed(), lo=lo, hi=hi), None))
    # root-box misses (emitted at refill time) alternating with rays that start inside the box
    alt = H.random_rays(4096, seed=seed(), lo=lo, hi=hi)
    alt[1::2] = _away_rays(rng, lo, hi, 2048)
    sets.append(("miss_alternating", alt, None))
    # a few whole-tree walkers among short rays
    mix = H.random_rays(2048, seed=seed(), lo=lo, hi=hi, tmax=f32(0.02) * diag)
    for k in (3, 700, 701, 2047):
        mix[k] = _nan_rays(1)[0]
    sets.append(("nan_mix", mix, None))
    sets.append(("indirect", H.random_rays(5000, seed=seed(), lo=lo - pad, hi=hi + pad), 3333))
    if lv is not None:
        sets.append(("comb", comb_rays(rng, lv), None))
    return [(s, np.ascontiguousarray(r), k) for s, r, k in sets]


def _scheduler_scenes():
    from tracer_b200 import harness as H
    comb, _, lv = comb_prim(MAX_DEPTH, interior_left=True, how="random", seed=5)
    prims = {"soup": _soup(), "c1": H.scene_c1(), "cornell": H.scene_reference_cornell(), "comb31": comb}
    cases = {k: _ray_sets(k, p, lv if k == "comb31" else None) for k, p in prims.items()}
    return prims, cases


def _trace_all(prims, cases):
    """Every case through both launch configurations (where usable), closest and any hit, trq_hit and trq_hit16.
    -> {key: record bytes}; indirect outputs are pre-filled with 0xFF so that records past *count show."""
    torch = _torch()
    from tracer_b200 import Scene, rays_to_torch
    from tracer_b200._lib import TrqError
    out = {}
    for sname, prim in prims.items():
        scene = Scene(prim, 0)
        for c in (0, 1):
            try:
                staged = scene.set_kernel_config(c)
            except TrqError:
                continue
            out[f"{sname}/cfg{c}/staged"] = np.array([staged], dtype=np.uint32)
            for rname, rays, count in cases[sname]:
                d = rays_to_torch(rays, "cuda:0")
                for a in (False, True):
                    for h16 in (False, True):
                        if count is None:
                            h = scene.hit(d, any=a, hit16=h16)
                        else:
                            h = torch.empty((rays.size, 4 if h16 else 8), dtype=torch.float32, device="cuda:0")
                            h.view(torch.int32).fill_(-1)
                            cnt = torch.tensor([count], dtype=torch.int64, device="cuda:0")
                            scene.hit_indirect(d, cnt, any=a, out=h, hit16=h16)
                        out[f"{sname}/{rname}/cfg{c}/any{int(a)}/{'h16' if h16 else 'h32'}"] = h.cpu().numpy().view(np.uint8).reshape(-1)
        scene.close()
    return out


def _save_inputs(path, prims, cases):
    z = {}
    for s, p in prims.items():
        for f in PRIM_FIELDS:
            z[f"prim/{s}/{f}"] = getattr(p, f)
    for s, lst in cases.items():
        for r, rays, count in lst:
            z[f"rays/{s}/{r}"] = rays
            z[f"count/{s}/{r}"] = np.array([-1 if count is None else count], dtype=np.int64)
    np.savez(path, **z)


def _load_inputs(path):
    from tracer_b200.scene import Primitive
    z = np.load(path)
    names = sorted({k.split("/")[1] for k in z.files if k.startswith("prim/")})
    prims = {s: Primitive(**{f: z[f"prim/{s}/{f}"] for f in PRIM_FIELDS}) for s in names}
    cases = {s: [] for s in names}
    for k in z.files:
        if k.startswith("rays/"):
            _, s, r = k.split("/")
            cnt = int(z[f"count/{s}/{r}"][0])
            cases[s].append((r, z[k], None if cnt < 0 else cnt))
    return prims, cases


def _worker_env(extra):
    env = {k: v for k, v in os.environ.items() if k not in KNOBS}
    env.update(extra)
    env["PYTHONPATH"] = ROOT + (os.pathsep + env["PYTHONPATH"] if env.get("PYTHONPATH") else "")
    return env


def _run_worker(mode, inp, out, env):
    p = subprocess.run([sys.executable, "-m", "tests.test_gpu_work_queue", mode, str(inp), str(out)], cwd=ROOT,
                       env=_worker_env(env), capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, f"worker {mode} {env}: rc {p.returncode}\n{p.stdout[-3000:]}\n{p.stderr[-3000:]}"


@pytest.fixture(scope="module")
def variants(built, tmp_path_factory):
    """Every compile-time variant, built in parallel (tools/build_variant.sh) into a temporary directory."""
    _torch()
    d = tmp_path_factory.mktemp("variants")
    env = dict(os.environ, TRQ_VARIANT_DIR=str(d))
    procs = {k: subprocess.Popen(["bash", os.path.join(ROOT, "tools", "build_variant.sh"), k, *flags], cwd=ROOT, env=env,
                                 stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for k, flags in VARIANTS.items()}
    libs = {}
    for k, p in procs.items():
        log, _ = p.communicate(timeout=1800)
        assert p.returncode == 0, f"variant {k}: {log[-3000:]}"
        libs[k] = str(d / f"libtracer_rq_{k}.so")
    return libs


def _first_difference(a, b, rec):
    if a.size != b.size:
        return f"{a.size} vs {b.size} bytes"
    bad = np.nonzero((a != b).reshape(-1, rec).any(axis=1))[0]
    return f"{bad.size} records differ, first {bad[:5].tolist()}"


def test_every_scheduler_setting_gives_the_default_bytes(built, port, variants, tmp_path):
    _torch()
    prims, cases = _scheduler_scenes()
    inp = tmp_path / "in.npz"
    _save_inputs(inp, prims, cases)
    default = _trace_all(prims, cases)
    # the default run against the oracle (once per case), and trq_hit16 as the packed form of trq_hit
    assert "c1/cfg1/staged" in default and int(default["c1/cfg1/staged"][0]) > 0
    assert "comb31/cfg1/staged" in default and "soup/cfg1/staged" in default and "cornell/cfg1/staged" in default
    for sname, prim in prims.items():
        for rname, rays, count in cases[sname]:
            live = rays if count is None else rays[:count]
            for a in (False, True):
                want, recs = oracle(port, prim, np.ascontiguousarray(live), a)
                for c in (0, 1):
                    if f"{sname}/cfg{c}/staged" not in default:
                        continue
                    key = f"{sname}/{rname}/cfg{c}/any{int(a)}"
                    h32 = default[key + "/h32"].view(L.hit_dtype)
                    h16 = default[key + "/h16"].view(L.hit16_dtype)
                    assert_hits_equal(h32[:live.size], want, key, recs)
                    assert np.array_equal(h16[:live.size].view(np.uint8), L.pack_hit16(h32[:live.size]).view(np.uint8)), key + " hit16"
                    if count is not None:
                        assert (h32[count:].view(np.uint8) == 0xFF).all() and (h16[count:].view(np.uint8) == 0xFF).all(), \
                            key + ": records written past *count"
    runs = [(name, env) for name, env in SETTINGS.items()]
    runs += [(name, {"TRQ_LIB": variants[name]}) for name in VARIANTS if name != "maxrays16"]

    def one(run):
        name, env = run
        out = tmp_path / f"{name}.npz"
        _run_worker("worker", inp, out, env)
        return name, out

    failures = []
    with ThreadPoolExecutor(max_workers=3) as ex:
        for name, out in ex.map(one, runs):
            got = np.load(out)
            if sorted(got.files) != sorted(default):
                failures.append(f"{name}: cases {sorted(set(default) ^ set(got.files))[:6]}")
                continue
            for k, v in default.items():
                if not np.array_equal(got[k], v):
                    failures.append(f"{name}: {k}: {_first_difference(got[k], v, 16 if k.endswith('h16') else 32)}")
    assert not failures, "\n".join(failures[:40])


# ------------------------------------------------------------------------------------------------------ staged prefixes
def test_every_staged_prefix_size_matches_the_oracle(soup, port):
    """TRQ_TOP_NODES (read per scene) caps the staged top-of-tree block: configuration 1 stages min(value, what fits)
    nodes -- a prefix that ends partway through a level, or the root alone -- and is refused with 0."""
    _torch()
    from tracer_b200 import Scene, harness as H
    from tracer_b200._lib import TrqError
    prim = soup
    plain = Scene(prim, 0)
    assert plain.info["topNodes"] == 2047
    fits = plain.set_kernel_config(1)
    plain.close()
    assert 0 < fits <= 2047
    rng = np.random.default_rng(7)
    rays = np.ascontiguousarray(np.concatenate([H.random_rays(60000, seed=71), adversarial_rays(rng, prim, 8000)]))
    short = rays.copy()
    short["tmax"] = f32(0.05)
    want = {False: oracle(port, prim, rays), True: oracle(port, prim, short, True)}
    for value in (0, 1, 2, 3, 7, 100, 2046, 2047):
        os.environ["TRQ_TOP_NODES"] = str(value)
        try:
            scene = Scene(prim, 0)
        finally:
            del os.environ["TRQ_TOP_NODES"]
        if value == 0:
            with pytest.raises(TrqError):
                scene.set_kernel_config(1)
        else:
            assert scene.set_kernel_config(1) == min(value, fits), value
            assert_hits_equal(gpu_trace(scene, rays, False), want[False][0], f"TRQ_TOP_NODES={value} closest", want[False][1])
            assert_hits_equal(gpu_trace(scene, short, True), want[True][0], f"TRQ_TOP_NODES={value} any", want[True][1])
        scene.close()


# ------------------------------------------------------------------------------------------------- split of large batches
SPLIT_N = 3 * (1 << 16) + 5


def _split_scene():
    from tracer_b200 import harness as H
    return H.scene_soup(20000, seed=3, extent=0.05), H.random_rays(SPLIT_N, seed=41)


def _split_outputs(scene, rays):
    """The calls whose batches a 2^16-ray launch limit splits (one timed launch per sub-batch)."""
    torch = _torch()
    from tracer_b200 import launch_count, rays_to_torch
    d = rays_to_torch(rays, "cuda:0")
    out = {}
    for name, kw in (("closest", {}), ("any", {"any": True}), ("hit16", {"hit16": True}), ("sorted", {"sort": True}),
                     ("reflayout", {"reflayout": True})):
        out[name] = scene.hit(d, **kw).cpu().numpy().view(np.uint8).reshape(-1)
    scene.profile(True)
    before = launch_count()
    scene.hit(d, sort=False)
    torch.cuda.synchronize()
    out["launches"] = np.array([launch_count() - before, scene.profile_read()[0]], dtype=np.int64)
    scene.profile(False)
    return out


def test_batches_past_the_launch_limit_are_split(built, port, variants, tmp_path):
    """A variant built with TRQ_MAX_RAYS_PER_LAUNCH = 2^16 traces 3 * 2^16 + 5 rays as four launches and gives the
    product library's bytes (one launch) for closest, any, trq_hit16, sorted and reference-layout traces; its
    trq_trace_indirect refuses a capacity above its limit."""
    _torch()
    from tracer_b200 import Scene
    prim, rays = _split_scene()
    scene = Scene(prim, 0)
    want = _split_outputs(scene, rays)
    scene.close()
    assert want["launches"].tolist() == [1, 1]
    sub = np.arange(0, SPLIT_N, 61)
    assert_like_oracle(want["closest"].view(L.hit_dtype)[sub], port, prim, np.ascontiguousarray(rays[sub]), False, "product")
    out = tmp_path / "split.npz"
    _run_worker("split", tmp_path / "unused", out, {"TRQ_LIB": variants["maxrays16"]})
    got = np.load(out)
    assert got["launches"].tolist() == [4, 4]
    assert int(got["indirect_rc"][0]) < 0
    for k in ("closest", "any", "hit16", "sorted", "reflayout"):
        assert np.array_equal(got[k], want[k]), f"{k}: {_first_difference(got[k], want[k], 16 if k == 'hit16' else 32)}"


def test_launch_size_limits_are_refused(built):
    """trq_trace_indirect covers its whole capacity with one launch, so a capacity above 2^31 is refused even when the
    device-resident count is small; a gather's capacity (and so a trq_trace_gather batch) is at most 2^31 rays."""
    torch = _torch()
    import ctypes as C
    from tracer_b200 import Scene, harness as H
    from tracer_b200._lib import lib
    scene = Scene(H.scene_soup(2000, seed=4, extent=0.05), 0)
    rays = torch.zeros((64, 8), dtype=torch.float32, device="cuda:0")
    hits = torch.zeros((64, 8), dtype=torch.float32, device="cuda:0")
    count = torch.tensor([3], dtype=torch.int64, device="cuda:0")
    rc = lib.trq_trace_indirect(scene._h, rays.data_ptr(), count.data_ptr(), (1 << 31) + 1, 0, hits.data_ptr(), None)
    assert rc < 0 and b"2^31" in lib.trq_last_error_string()
    g, handle = C.c_void_p(), C.create_string_buffer(64)
    rc = lib.trq_gather_create(scene._h, 0, 1, (1 << 31) + 1, C.byref(g), handle)
    assert rc < 0 and not g.value and b"capacity" in lib.trq_last_error_string()
    torch.cuda.synchronize()
    assert (hits == 0).all()
    scene.close()


GIB = 1 << 30


def test_more_than_2_31_rays(built, port):
    """n = 2^31 + 4097 rays built on the device as base[i % M] (M prime, base checked against the oracle): every record
    equals the base's, on both sides of the 2^31 boundary and at the last ray; two launches. n = 2^31 is one launch.
    Needs about 100 GiB of free device memory (the GPU may be shared): 64 GiB of rays, 32 GiB of trq_hit16 records;
    trq_hit records and the sorted path run only when there is room for them as well."""
    torch = _torch()
    from tracer_b200 import Scene, harness as H, launch_count, rays_to_torch
    free = torch.cuda.mem_get_info()[0]
    n, M = (1 << 31) + 4097, 999983
    if free < 100 * GIB:
        pytest.skip(f"{free / GIB:.0f} GiB of device memory free, about 100 GiB needed for 2^31 + 4097 rays")
    prim = H.scene_soup(20000, seed=6, extent=0.05)
    base_h = H.random_rays(M, seed=61)
    scene = Scene(prim, 0)
    base = rays_to_torch(base_h, "cuda:0")
    want16 = scene.hit(base, hit16=True, sort=False)
    want32 = scene.hit(base, sort=False)
    sub = np.concatenate([np.arange(0, M, 101), [M - 1]])
    assert_like_oracle(want32.cpu().numpy().view(L.hit_dtype).reshape(-1)[sub], port, prim, np.ascontiguousarray(base_h[sub]),
                       False, "base")
    chunk = 1 << 26
    rays = torch.empty((n, 8), dtype=torch.float32, device="cuda:0")
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        rays[lo:hi] = base[torch.arange(lo, hi, device="cuda:0") % M]

    def check(hits, want, m, where):
        for lo in range(0, m, chunk):
            hi = min(m, lo + chunk)
            ok = torch.equal(hits[lo:hi].view(torch.int32), want[torch.arange(lo, hi, device="cuda:0") % M].view(torch.int32))
            assert ok, f"{where}: records [{lo}, {hi}) differ"
        for i in (m - 1, (1 << 31) - 1, 1 << 31):                # the last ray, and both sides of 2^31
            if i < m:
                assert torch.equal(hits[i].view(torch.int32), want[i % M].view(torch.int32)), f"{where}: ray {i}"

    def run(m, hit16, sort, launches):
        hits = torch.empty((m, 4 if hit16 else 8), dtype=torch.float32, device="cuda:0")
        hits.view(torch.int32).fill_(-1)
        before = launch_count()
        scene.hit(rays[:m], hit16=hit16, sort=sort, out=hits)
        torch.cuda.synchronize()
        where = f"n={m} hit16={hit16} sort={sort}"
        if launches is not None:
            assert launch_count() - before == launches, where
        check(hits, want16 if hit16 else want32, m, where)
        del hits
        torch.cuda.empty_cache()

    run(n, True, False, 2)
    run(1 << 31, True, False, 1)
    skipped = []
    if torch.cuda.mem_get_info()[0] >= 70 * GIB:
        run(n, False, False, 2)
    else:
        skipped.append("trq_hit records (64 GiB)")
    if torch.cuda.mem_get_info()[0] >= 54 * GIB:
        run(n, True, True, None)                               # + ordering passes; 16 GiB of stream-ordered scratch
    else:
        skipped.append("sort=True (32 GiB of records + 16 GiB of scratch)")
    if skipped:
        print("not run for lack of device memory: " + "; ".join(skipped))
    del rays
    scene.close()
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------- the workers
def _worker(inp, out):
    prims, cases = _load_inputs(inp)
    np.savez(out, **_trace_all(prims, cases))


def _split_worker(out):
    import ctypes as C  # noqa: F401
    import torch
    from tracer_b200 import Scene
    from tracer_b200._lib import lib
    prim, rays = _split_scene()
    scene = Scene(prim, 0)
    res = _split_outputs(scene, rays)
    d = torch.zeros((1 << 16) + 1, 8, dtype=torch.float32, device="cuda:0")
    cnt = torch.tensor([5], dtype=torch.int64, device="cuda:0")
    res["indirect_rc"] = np.array([lib.trq_trace_indirect(scene._h, d.data_ptr(), cnt.data_ptr(), d.shape[0], 0, d.data_ptr(), None)])
    scene.close()
    np.savez(out, **res)


if __name__ == "__main__":
    mode, inp, out = sys.argv[1:4]
    if mode == "worker":
        _worker(inp, out)
    elif mode == "split":
        _split_worker(out)
    else:
        raise SystemExit(f"unknown mode {mode}")
    print(json.dumps({"mode": mode, "out": out}))
