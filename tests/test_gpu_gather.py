"""Multi-GPU hit delivery against the oracle: the peer-memory gather (trq_trace_gather, both sender kernels, tile sizes 2^8,
2^11 and 2^16, every leaf specialisation) and the NCCL chunked all-gather (dist.trace_and_gather).

A torchrun worker traces four scenes in one process per rank, twelve steps each, with step sizes at the edges of a tile
(T = 2^shift records) and of a 12 KB TMA chunk (C records) in both record formats. Every rank saves every slot it
received, so each size is checked after a sender kernel has shipped it to another rank. The parent regenerates
every rank's rays from their seeds and compares each received record with the oracle: ids and flags equal, t bit for
bit, u / v bit for bit except on sphere hits, which follow the sphere-uv rule of tests/test_gpu_special_rays.py. It also
reads which kernels ran (torch.profiler in the worker), so that the coverage the settings claim is checked, not assumed.
On a one-GPU box the ranks share device 0 (CUDA IPC between processes on one device, gloo rendezvous); with >= 2 GPUs
the default and LSU settings also run one rank per GPU over NCCL, and so does the trace_and_gather test."""
import os
import re
import socket
import subprocess
import sys
import time

import numpy as np
import pytest

from tracer_b200 import layout as L

from .test_special_rays_cpu import comb_right, nan_origin_rays
from .util import bits

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TMA_CHUNK = 12288                                      # TRQ_SEND_TMA_CHUNK: bytes per TMA bulk copy
CHUNK_RECORDS = {False: TMA_CHUNK // 32, True: TMA_CHUNK // 16}        # C: 384 trq_hit, 768 trq_hit16
# capacity per tile shift: >= 3T + 17, not a multiple of T (a partial last tile), >= 65536 so that sort=True orders the
# queue (the library sorts batches of 2^16 rays and more)
CAPACITY = {8: 70_001, 11: 100_003, 16: 200_003}
SCENES = ("soup", "cornell", "c1", "comb31")
# sender and tile settings of one worker run (the library reads both once per process)
SETTINGS = {
    "default": {},
    "lsu": {"TRQ_GATHER_TMA": "0"},
    "tile256": {"TRQ_GATHER_TILE_SHIFT": "8"},
    "tile65536": {"TRQ_GATHER_TILE_SHIFT": "16"},
    "tile256-lsu": {"TRQ_GATHER_TILE_SHIFT": "8", "TRQ_GATHER_TMA": "0"},
}


def build_scene(name):
    """soup: LEAVES_TRI. cornell: the reference's Cube + Square + Sphere + Triangle mix, LEAVES_ALL. c1: spheres only,
    LEAVES_TRI_SPHERE, whose automatic launch configuration is the staged 1024x1 one. comb31: the depth-31 comb, whose
    far-child stack leaves no room for the TMA sender's staging beside five trace CTAs."""
    from tracer_b200 import harness as H
    return {"soup": lambda: H.scene_soup(50_000, seed=1, extent=0.02), "cornell": H.scene_reference_cornell,
            "c1": H.scene_c1, "comb31": comb_right}[name]()


def scene_rays(name, prim, step, rank, n):
    """Rank `rank`'s n rays of step `step`: seeded random rays over the scene (disjoint streams per rank, a new seed per
    step, so that a stale phase or another rank's records cannot match). On the comb every 97th ray has a NaN origin
    (nan_origin_rays), which fills the far-child stack to its bound."""
    from tracer_b200 import harness as H
    if name == "c1":
        lo, hi = (-11.0, 0.0, -11.0), (11.0, 2.0, 11.0)        # the small spheres, not the ground sphere's box
    else:
        b = prim.bvhList
        fin = np.isfinite(b["mini"]).all(axis=1) & np.isfinite(b["maxi"]).all(axis=1)
        lo, hi = b["mini"][fin].min(axis=0), b["maxi"][fin].max(axis=0)
    rays = H.random_rays(n, seed=100 * (SCENES.index(name) + 1) + step, lo=lo, hi=hi, first=rank << 24)
    if name == "comb31" and n:
        rays[::97] = nan_origin_rays(np.random.default_rng([step, rank]), rays[::97].size)
    return rays


def step_plan(shift):
    """[(any, hit16, sort, (size of rank 0, 1, 2, 3))] for one worker run. Ranks 0 and 1 alone trace every size of
    edge_sizes in both record formats, so with two ranks each of them reaches the other rank through a sender kernel;
    ranks 2 and 3 add more ragged shards."""
    T, cap = 1 << shift, CAPACITY[shift]
    c32, c16 = CHUNK_RECORDS[False], CHUNK_RECORDS[True]
    return [
        (False, False, False, (cap, 0, T + 1, 5)),                   # trq_hit
        (False, False, True, (T - 1, cap, 1, 3 * T + 17)),
        (True, False, False, (c32 - 1, T, c32 + 1, 0)),
        (False, False, False, (1, 3 * T + 17, T - 1, c32)),
        (True, False, True, (c32, cap - 1, c32 - 1, cap)),
        (False, False, False, (T + 1, c32 + 1, 0, T)),
        (False, True, False, (c16 + 1, 3 * T + 17, c16, T - 1)),     # trq_hit16
        (True, True, True, (1, cap, c16 - 1, cap - 1)),
        (False, True, False, (c16, c16 - 1, T, 1)),
        (True, True, False, (T, 0, 3 * T + 17, c16 + 1)),
        (False, True, True, (cap - 1, T - 1, 1, cap)),
        (True, True, False, (T + 1, c16 + 1, 0, c16)),
    ]


def edge_sizes(shift, hit16):
    """The shard sizes every worker run must deliver in one record format: 0, 1, T - 1, T, T + 1, 3T + 17, the
    capacity, and C - 1, C, C + 1, where C records make one TMA chunk (a tile of C records is exactly one chunk)."""
    T, C = 1 << shift, CHUNK_RECORDS[hit16]
    return {0, 1, T - 1, T, T + 1, 3 * T + 17, CAPACITY[shift], C - 1, C, C + 1}


def expected_leaves(prim):
    """The LEAVES_* specialisation the library picks (trq_api.cu: from the leaf counts)."""
    if prim.sphereList.size + prim.squareList.size + prim.cubeList.size == 0:
        return 2                                                       # LEAVES_TRI
    return 1 if prim.squareList.size + prim.cubeList.size == 0 else 0  # LEAVES_TRI_SPHERE, LEAVES_ALL


# ----------------------------------------------------------------------------------------------------- oracle checks
_cache = {}


def _prim(name):
    if ("prim", name) not in _cache:
        _cache[("prim", name)] = build_scene(name)
    return _cache[("prim", name)]


def _oracle(port, prim, rays, any_hit):
    spheres = prim.sphereList.size > 0                                 # sphere uv needs the oracle's normals
    return port.trace(prim, rays, any=any_hit, records=spheres, nthreads=8)


def _differs(got, want, fields, uv_mask):
    """Per record: does any field differ from the oracle (bits, NaN-aware; u / v only where uv_mask)?"""
    bad = np.zeros(got.size, dtype=bool)
    for f in fields:
        a, b = got[f], want[f]
        same = (bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b)) if a.dtype.kind == "f" else a == b
        bad |= ~same if f not in ("u", "v") else (~same & uv_mask)
    return bad


def assert_slot(got_bytes, want, hit16, where):
    """One received slot against the oracle's records for the same rays. The message names the first bad index and
    whether the record there is all zero (never delivered) or another record (a stale phase, a wrong tile)."""
    from .test_gpu_special_rays import assert_sphere_uv
    hits = want["hits"]
    got = got_bytes.view(L.hit16_dtype if hit16 else L.hit_dtype)
    assert got.size == hits.size, f"{where}: {got.size} records, want {hits.size}"
    hit = (hits["flags"] & L.HIT_FLAG_HIT) != 0
    sph = hit & (hits["pType"] == L.SPHERE)
    if hit16:
        ref, fields = L.pack_hit16(hits), ("t", "id", "u", "v")
    else:
        ref, fields = hits, ("t", "pType", "pIndex", "leafNode", "material", "flags", "u", "v")
    bad = np.nonzero(_differs(got, ref, fields, ~sph))[0]
    if bad.size:
        i = int(bad[0])
        rec = got_bytes.reshape(got.size, -1)[i]
        what = ("all 0xff: never delivered (poison_phases filled it)" if (rec == 0xFF).all() else
                "all zero: a zeroed record" if not rec.any() else "a different record (a stale phase, another tile or rank)")
        raise AssertionError(f"{where}: {bad.size} of {got.size} records differ from the oracle, first at index {i}: {what}; "
                             f"got {got[i]} want {ref[i]}")
    if sph.any():
        rec = want["records"]
        assert_sphere_uv(got["u"][sph], got["v"][sph], rec["gn"][sph], hits["u"][sph], hits["v"][sph], where + " sphere uv")
    return int(hit.sum())


def check_worker_output(port, path, setting, world, shift, tma):
    """Everything one rank saved in one worker run (the files under `path`), against the oracle. Returns a summary line."""
    plan = step_plan(shift)
    lines = []
    for name in SCENES:
        prim = _prim(name)
        z = np.load(os.path.join(path, f"{name}.npz"))
        saver = int(z["rank"])
        hits_seen = 0
        for k, (any_hit, hit16, sort, sizes) in enumerate(plan):
            ns = list(sizes[:world])
            where = (f"[{setting}] {name} step {k} ({'any' if any_hit else 'closest'} hit, {'trq_hit16' if hit16 else 'trq_hit'}"
                     f"{', sort' if sort else ''})")
            counts = z[f"counts{k}"].tolist()
            assert counts == ns, f"{where}: rank {saver} received counts {counts}, the ranks traced {ns}"
            for r in range(world):
                rays = scene_rays(name, prim, k, r, ns[r])
                key = (name, k, r, ns[r], any_hit)
                if key not in _cache:
                    _cache[key] = _oracle(port, prim, rays, any_hit)
                hits_seen += assert_slot(z[f"step{k}_slot{r}"], _cache[key], hit16, f"{where} slot {r} on rank {saver}")
        assert hits_seen > 0, f"[{setting}] {name}: no hit among the received records: the comparison would prove nothing"
        lines.append(f"{name}: {hits_seen} hits")
        if "kernels" not in z:
            continue
        # which kernels ran (rank 0's step 0, which traces the capacity): the sender the settings select, configuration 0
        # (256 threads x 5 CTAs, nothing staged) under every gather, and the leaf specialisation of the scene
        kernels = [str(s) for s in z["kernels"]]
        senders = {s for s in ("gather_send_tma_kernel", "gather_send_kernel") if any(s + "(" in k or s + "<" in k or k.endswith(s) for k in kernels)}
        want_sender = "gather_send_tma_kernel" if tma and name != "comb31" else "gather_send_kernel"
        assert senders == {want_sender}, f"[{setting}] {name}: sender kernels {senders}, want {want_sender} (kernels seen: {kernels})"
        traced = {m.groups() for k in kernels for m in re.finditer(r"trace_packed_kernel<(\w+), (\d+), (\d+), (\d+), (\w+), (\d+)>", k)}
        assert traced, f"[{setting}] {name}: no traversal kernel among {kernels}"
        for any_t, out, block, minb, top, leaves in traced:
            assert (block, minb, top) == ("256", "5", "false"), f"[{setting}] {name}: a gather traced with {block}x{minb} top={top}"
            assert int(leaves) == expected_leaves(prim), f"[{setting}] {name}: leaf specialisation {leaves}"
        if name == "c1":                                               # trq_trace alone would use the staged configuration
            assert str(z["auto_cfg"]).startswith("1024x1"), f"[{setting}] c1: automatic configuration {z['auto_cfg']}"
        lines[-1] = f"{name}: {want_sender}, cfg 256x5 (trq_trace: {z['auto_cfg']}), depth {int(z['depth'])}, {hits_seen} hits"
    return f"rank {saver}: " + "; ".join(lines)


# ------------------------------------------------------------------------------------------------------------ worker
WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["TRQ_ROOT"])
import numpy as np, torch
from tracer_b200 import Scene, dist as D, rays_to_torch
from tests import test_gpu_gather as T
shared = os.environ["TRQ_SHARE_DEVICE"] == "1"
rank, local_rank, world = D.init(backend="gloo" if shared else None)
local_rank = 0 if shared else local_rank
torch.cuda.set_device(local_rank)
dev = f"cuda:{local_rank}"
out = os.environ["TRQ_OUT"]
save = True                                                       # every rank: each slot it receives comes through a sender

if os.environ["TRQ_MODE"] == "peer":
    shift = int(os.environ.get("TRQ_GATHER_TILE_SHIFT", "11"))
    cap = T.CAPACITY[shift]
    for name in T.SCENES:
        prim = D.replicate_primitive(T.build_scene(name) if rank == 0 else None, src=0)
        scene = Scene(prim, local_rank)
        g = D.HitGather(scene, cap)
        T.poison_phases(g, D.barrier)
        saved, prev = {}, None
        for k, (any_hit, hit16, sort, sizes) in enumerate(T.step_plan(shift)):
            ns = list(sizes[:world])
            mine = rays_to_torch(T.scene_rays(name, prim, k, rank, ns[rank]), dev) if ns[rank] else torch.empty((0, 8), device=dev)
            prof = torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) if k == 0 and rank == 0 else None
            if prof: prof.start()
            g.trace(mine, any=any_hit, hit16=hit16, sort=sort)
            hits_all, counts = g.wait()
            torch.cuda.synchronize()
            if prof:
                prof.stop()
                saved["kernels"] = np.array(sorted({e.key for e in prof.key_averages() if "kernel" in e.key}))
            g.status()
            got = [hits_all[r, :ns[r]].cpu() for r in range(world)]
            if prev is not None:                                  # the previous step's result is still intact (three phases)
                p_all, p_got, p_ns = prev
                for r in range(world):
                    assert torch.equal(p_all[r, :p_ns[r]].cpu().view(torch.int32), p_got[r].view(torch.int32)), f"{name} step {k}: step {k - 1} slot {r} changed"
            prev = (hits_all, got, ns)
            if save:
                saved[f"counts{k}"] = counts.cpu().numpy()
                for r in range(world):
                    saved[f"step{k}_slot{r}"] = got[r].numpy().view(np.uint8).reshape(-1)
            D.barrier()                                           # nobody starts step k+1 before everybody checked step k-1
        g.status()
        if save:
            np.savez(os.path.join(out, f"rank{rank}", f"{name}.npz"), rank=rank, auto_cfg=scene.kernel_config(),
                     depth=scene.info["maxDepth"], **saved)
        g.close()
        scene.close()
else:                                                             # dist.trace_and_gather, every rank the same n
    prim = D.replicate_primitive(T.build_scene("soup") if rank == 0 else None, src=0)
    scene = Scene(prim, local_rank)
    saved = {}
    for n, chunks in T.TAG_CASES:
        for any_hit in (False, True):
            mine = rays_to_torch(T.scene_rays("soup", prim, 90 + any_hit, rank, n), dev)
            local = torch.full((n, 8), -7.0, device=dev)
            hits_all = torch.full((world, n, 8), -7.0, device=dev)
            D.trace_and_gather(scene, mine, local, hits_all, any=any_hit, sort=True, chunks=chunks)
            torch.cuda.synchronize()
            for r in range(world):                                # rank r's rays traced here in full: identical bytes
                want = scene.hit(rays_to_torch(T.scene_rays("soup", prim, 90 + any_hit, r, n), dev), any=any_hit)
                assert torch.equal(hits_all[r].view(torch.int32), want.view(torch.int32)), f"trace_and_gather n={n} any={any_hit}: slot {r} on rank {rank}"
            assert torch.equal(local.view(torch.int32), hits_all[rank].view(torch.int32))
            if save:
                sub = T.tag_subsample(n)
                for r in range(world):
                    saved[f"n{n}_any{int(any_hit)}_slot{r}"] = hits_all[r][torch.from_numpy(sub).to(dev)].cpu().numpy().view(np.uint8).reshape(-1)
    if save:
        np.savez(os.path.join(out, f"rank{rank}", "tag.npz"), **saved)
    scene.close()
D.barrier()
os.write(1, f"rank {rank} ok\n".encode())                     # one write: the ranks share the pipe
'''

TAG_CASES = ((3, 4), (1, 4), (1_000_003, 4))                  # n = 3 in 4 chunks: one chunk is empty and skipped


def poison_phases(g, barrier=lambda: None):
    """Three empty steps, one per buffer phase, each followed by filling every slot of this rank's buffer with 0xff
    bytes (a NaN t, flags 0xffffffff): a record that is never delivered cannot pass for a miss. The barrier keeps
    every rank's fill before any rank's next step."""
    import torch
    for _ in range(3):
        g.trace(torch.empty((0, 8), dtype=torch.float32, device=f"cuda:{g.scene.device}"))
        hits_all, counts = g.wait()
        torch.cuda.synchronize()
        g.status()
        assert counts.tolist() == [0] * g.world
        hits_all.view(torch.int32).fill_(-1)
        torch.cuda.synchronize()
        barrier()


def tag_subsample(n):
    return np.unique(np.concatenate([np.arange(0, n, 997), [n - 1]]))


def _run_worker(tmp_path, world, shared, mode, env_extra):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    for r in range(world):
        (tmp_path / f"rank{r}").mkdir(exist_ok=True)
    env = {k: v for k, v in os.environ.items() if not k.startswith("TRQ_GATHER_")}
    env.update(env_extra, TRQ_ROOT=ROOT, TRQ_OUT=str(tmp_path), TRQ_MODE=mode, TRQ_SHARE_DEVICE="1" if shared else "0")
    t0 = time.time()
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
                       env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=900)
    out = p.stdout.decode()
    assert p.returncode == 0, out[-6000:]
    for r in range(world):
        assert f"rank {r} ok" in out, out[-6000:]
    return time.time() - t0


def _peer_run(port, tmp_path, capsys, setting, world, shared):
    env = SETTINGS[setting]
    dt = _run_worker(tmp_path, world, shared, "peer", env)
    shift = int(env.get("TRQ_GATHER_TILE_SHIFT", "11"))
    tma = env.get("TRQ_GATHER_TMA", "1") != "0"
    for hit16 in (False, True):                    # every edge size is traced by a rank whose records another rank checks
        traced = {sizes[r] for _, h, _, sizes in step_plan(shift) if h == hit16 for r in range(world)}
        assert edge_sizes(shift, hit16) <= traced, sorted(edge_sizes(shift, hit16) - traced)
    summary = [check_worker_output(port, str(tmp_path / f"rank{r}"), setting, world, shift, tma) for r in range(world)]
    with capsys.disabled():
        where = "on device 0" if shared else "one per GPU (NCCL)"
        print(f"\ngather worker [{setting}] tile 2^{shift}, {world} ranks {where}: {dt:.1f} s; " + " | ".join(summary))


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.mark.parametrize("setting", list(SETTINGS))
def test_peer_gather_two_ranks_on_one_gpu(built, port, tmp_path, capsys, setting):
    """Runs wherever there is a GPU: two processes share device 0."""
    _torch()
    _peer_run(port, tmp_path, capsys, setting, 2, shared=True)


@pytest.mark.parametrize("setting", ["default", "lsu"])
def test_peer_gather_one_rank_per_gpu(built, port, tmp_path, capsys, setting):
    """The NVLink path: one rank per GPU (up to 4) over NCCL."""
    torch = _torch()
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs (one rank per GPU); the two-ranks-on-one-GPU runs cover the protocol")
    _peer_run(port, tmp_path, capsys, setting, min(torch.cuda.device_count(), 4), shared=False)


# ------------------------------------------------------------------------------------------------ in-process tests
def _gather_step(g, rays, any_hit=False, hit16=False, sort=False):
    torch = _torch()
    g.trace(rays, any=any_hit, hit16=hit16, sort=sort)
    hits_all, counts = g.wait()
    torch.cuda.synchronize()
    g.status()
    return hits_all, counts


def test_one_rank_gather(built, port):
    """HitGather without a process group (world 1, no peer): slot 0 holds the oracle's records, both formats."""
    _torch()
    from tracer_b200 import Scene, dist as D, rays_to_torch
    prim = _prim("cornell")
    scene = Scene(prim, 0)
    cap = CAPACITY[11]
    g = D.HitGather(scene, cap)
    assert g.world == 1
    poison_phases(g)
    for k, n in enumerate((0, 1, 383, 384, 385, 767, 768, 769, 2047, 2048, 2049, 6161, cap)):
        any_hit, hit16, sort = k % 3 == 1, k % 2 == 1, n == cap
        rays = scene_rays("cornell", prim, 50 + k, 0, n)
        hits_all, counts = _gather_step(g, rays_to_torch(rays, "cuda:0"), any_hit, hit16, sort)
        assert counts.tolist() == [n]
        got = hits_all[0, :n].cpu().numpy().view(np.uint8).reshape(-1)
        assert_slot(got, _oracle(port, prim, rays, any_hit), hit16, f"one rank n={n} any={any_hit} hit16={hit16}")
    g.close()
    scene.close()


def test_connected_gather_refuses_bad_arguments(built, port):
    """A connected gather refuses, with a negative status and a message and without advancing its step: trq_gather_wait
    before any trace, more rays than the capacity, host pointers, the reference-layout kernel, rays 16 bytes off their
    32-byte alignment, NULL rays, another scene's handle, and a second trq_gather_connect. The next valid step still
    gives the oracle's records."""
    torch = _torch()
    import ctypes as C
    from tracer_b200 import Scene, dist as D, rays_to_torch
    from tracer_b200._lib import lib
    prim = _prim("soup")
    scene, other = Scene(prim, 0), Scene(_prim("comb31"), 0)
    cap = 5000
    g = D.HitGather(scene, cap)
    hp, cp = C.c_void_p(), C.c_void_p()
    assert lib.trq_gather_wait(g._h, None, C.byref(hp), C.byref(cp)) < 0
    assert b"nothing traced" in lib.trq_last_error_string()
    poison_phases(g)
    n = 4000
    host = scene_rays("soup", prim, 60, 0, n)
    rays = rays_to_torch(host, "cuda:0")
    over = rays_to_torch(scene_rays("soup", prim, 61, 0, cap + 1), "cuda:0")
    padded = torch.zeros((n + 1, 8), dtype=torch.float32, device="cuda:0")
    padded.view(-1)[4:4 + 8 * n] = rays.view(-1)                      # the same rays, starting 16 bytes in
    st = torch.cuda.current_stream().cuda_stream
    cases = (("more rays than the capacity", scene, over.data_ptr(), cap + 1, 0, b"capacity"),
             ("TRQ_HOST_PTRS", scene, host.ctypes.data, n, L.HOST_PTRS, b"device pointers"),
             ("TRQ_HOST_ASYNC", scene, rays.data_ptr(), n, L.HOST_ASYNC, b"device pointers"),
             ("TRQ_KERNEL_REFLAYOUT", scene, rays.data_ptr(), n, L.KERNEL_REFLAYOUT, b"packed kernel"),
             ("rays offset by 16 bytes", scene, padded.data_ptr() + 16, n, 0, b"aligned"),
             ("NULL rays", scene, None, n, 0, b"NULL rays"),
             ("another scene", other, rays.data_ptr(), n, 0, b"foreign"))
    want = {a: _oracle(port, prim, host, a) for a in (False, True)}
    for k, (what, s, ptr, cnt, flags, msg) in enumerate(cases):
        rc = lib.trq_trace_gather(s._h, g._h, ptr, cnt, flags, st)
        assert rc < 0, f"{what}: status {rc}"
        assert msg in lib.trq_last_error_string(), f"{what}: {lib.trq_last_error_string()}"
        hits_all, counts = _gather_step(g, rays, any_hit=k % 2 == 1)
        assert counts.tolist() == [n], what
        assert_slot(hits_all[0, :n].cpu().numpy().view(np.uint8).reshape(-1), want[k % 2 == 1], False, f"after refusing {what}")
    handle = C.create_string_buffer(64)
    assert lib.trq_gather_connect(g._h, handle) < 0
    assert b"already connected" in lib.trq_last_error_string()
    hits_all, counts = _gather_step(g, rays, hit16=True)
    assert_slot(hits_all[0, :n].cpu().numpy().view(np.uint8).reshape(-1), want[False], True, "after a second connect")
    g.close()
    other.close()
    scene.close()


def test_trace_and_gather_world_one(built, port):
    """dist.trace_and_gather without a process group: hits_all[0] and hits_local both equal the oracle."""
    torch = _torch()
    from tracer_b200 import Scene, dist as D, rays_to_torch
    prim = _prim("soup")
    scene = Scene(prim, 0)
    for n, any_hit, sort in ((1, False, False), (70_001, True, True), (200_003, False, True)):
        rays = scene_rays("soup", prim, 70, 0, n)
        local = torch.full((n, 8), -7.0, device="cuda:0")
        hits_all = torch.full((1, n, 8), -7.0, device="cuda:0")
        D.trace_and_gather(scene, rays_to_torch(rays, "cuda:0"), local, hits_all, any=any_hit, sort=sort)
        torch.cuda.synchronize()
        want = _oracle(port, prim, rays, any_hit)
        for what, t in (("hits_all[0]", hits_all[0]), ("hits_local", local)):
            assert_slot(t.cpu().numpy().view(np.uint8).reshape(-1), want, False, f"trace_and_gather world 1 n={n}: {what}")
    scene.close()


def test_trace_and_gather_across_ranks(built, port, tmp_path):
    """dist.trace_and_gather over NCCL, every rank the same n (3 in 4 chunks, 1, 1 000 003), closest and any hit,
    sort=True: each rank checks every hits_all[r] against a local trace of rank r's rays in full; here rank 0's copy is
    checked against the oracle on a subsample."""
    torch = _torch()
    if torch.cuda.device_count() < 2:
        pytest.skip("NCCL needs one rank per GPU: this box has one GPU (the world-size-1 path is tested above)")
    world = min(torch.cuda.device_count(), 4)
    _run_worker(tmp_path, world, False, "tag", {})
    prim = _prim("soup")
    z = np.load(str(tmp_path / "rank0" / "tag.npz"))
    for n, _ in TAG_CASES:
        sub = tag_subsample(n)
        for any_hit in (False, True):
            for r in range(world):
                rays = scene_rays("soup", prim, 90 + any_hit, r, n)[sub]
                assert_slot(z[f"n{n}_any{int(any_hit)}_slot{r}"], _oracle(port, prim, rays, any_hit), False,
                            f"trace_and_gather n={n} any={any_hit} slot {r} on rank 0")
