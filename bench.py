#!/usr/bin/env python
"""bench.py -- headline benchmark of the ray-query hot path (contract: see DESIGN.md section 6).

    python bench.py --gpus N --steps K --warmup W [--workload c3|c1|c2|c4|c5|soup1m|...] [--impl reference]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path (trq_trace) over one batch of synthetic rays of the named BASELINE config.
Every timed region runs exactly K steps. --dump-outputs writes what the last timed step returned (see dump_outputs).
Default workload = C3 (the config the north_star target is quoted on): the ~1.0 M-triangle "meshes" scene (coatball +
teapot subdivided twice inside the Cornell box) traced with the incoherent diffuse-bounce rays spawned from the
3840x2160 primary hits. The default run also measures BASELINE.json's other configs (`workloads`: c1, c2, c4, c5).

  value     whole-job Mrays/s, rays and hit buffers resident in HBM, CUDA events, max over ranks
  e2e       the same metric through the C-ABI with HOST buffers (pinned), H2D + D2H inside the timed region
  roofline  traversal kernel only: algorithmic bytes (instrumented-oracle step counts, SURVEY 8d formula) / its
            CUDA-event duration, against the ceiling that bounds the workload: L2 bandwidth for scenes that live in
            L2 (C1-C4), HBM bandwidth for those that do not (C5, soups); the DRAM share is reported beside it
  cpu_baseline  the reference's own Scene::hit (oracle/_ref, compiled verbatim) on the host cores, on a
            bounded strided sample of the same rays (N=1, rank 0 only)

`--impl reference` times that CPU reference alone (rank 0; other ranks exit).
Multi-GPU: one process per GPU (torchrun), scene broadcast from rank 0 over NCCL, rays sharded by batch (weak scaling:
each rank traces its own batch; C5 is the fixed 64 M-ray frame cut N ways), no collective on the data path;
`with_hit_allgather` adds the figure with every rank's records delivered to every rank (trq_trace_gather).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Mrays/sec closest-hit"
UNIT = "Mrays/s"
HBM_FALLBACK_GBS = 6650.0
C5_FRAME_RAYS = 64_000_000

WORKLOADS = {
    "c2": "C2: RT_Metal Cornell box triangles + teapot (15.7k tris), 1920x1080 primary + 1 diffuse bounce, device-resident wavefront (cast, trace, spawn, trace)",
    "c2bounce": "C2 geometry, only the diffuse bounce batch spawned from the 1920x1080 primary hits",
    "c3path": "C3 geometry (1.0M tris), 3840x2160 primary + 1 diffuse bounce, device-resident wavefront (cast, trace, spawn, trace)",
    "c3": "C3: RT_Metal meshes scene (coatball+teapot subdivided x16, 1.0M tris), incoherent diffuse bounce rays from 3840x2160 primary hits",
    "c4": "C4: C3 geometry + 10,012 spheres, any-hit shadow rays toward light squares 5/6 from 3840x2160 primary hits",
    "c5": "C5: 10M-triangle random soup, 64M uniform incoherent rays per frame, the frame sharded by ray batch over the GPUs",
    "soup1m": "1M-triangle random soup, 8M uniform incoherent rays",
    "c1": "C1: RT_Nextweek randomScene (442 spheres) as Sphere leaves of the RT_Metal SAH BVH, 1280x720 primary rays (camera0)",
}
# the memory level that bounds the traversal kernel: scenes whose packed working set lives in the 126 MB L2 -> "l2";
# scenes that do not fit -> "hbm" (SURVEY 8d)
BOUND = {"c1": "l2", "c2": "l2", "c2bounce": "l2", "c3": "l2", "c3path": "l2", "c4": "l2", "c5": "hbm", "soup1m": "hbm"}
EXTRA_WORKLOADS = ("c1", "c2", "c4", "c5")          # measured by the default run next to the main workload
# device-resident wavefronts: name -> image size (primary rays per step); the Cornell camera of Tracer.mm:371-411
PATH_WORKLOADS = {"c2": (1920, 1080), "c3path": (3840, 2160)}
# algorithmic bytes per ray measured once by the instrumented oracle (DESIGN.md section 4); used only if the
# oracle cannot be run in this process. Recomputed live on a sample otherwise.
BYTES_PER_RAY_FALLBACK = {"c3path": 1400.0, "c2bounce": 1094.0, "c1": 700.0, "c2": 1094.0, "c3": 1778.0, "c4": 2887.0, "c5": 9184.0, "soup1m": 7039.0}
DUMP_BYTES = 60_000_000        # --dump-outputs writes at most this much: kept small enough to store and diff two runs


def L_ray_dtype():
    from tracer_b200 import layout
    return layout.ray_dtype


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


def traffic_table():
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(tp))
    except Exception:
        return {}


# ----------------------------------------------------------------------------------------------- workloads
def build_scene(name):
    from tracer_b200 import harness as H
    if name in ("c2", "c2bounce"):
        return H.scene_c2()
    if name in ("c3", "c3path"):
        return H.scene_c3(2)
    if name == "c4":
        return H.scene_c4(2)
    if name == "c5":
        return H.scene_soup(10_000_000, seed=1, extent=0.004)
    if name == "soup1m":
        return H.scene_soup(1_000_000, seed=1, extent=0.01)
    if name == "c1":
        return H.scene_c1()
    raise SystemExit(f"unknown workload {name}")


def c1_rays():
    """RT_Nextweek camera0 (Render.swift:35-57): from (13,2,3) to the origin, vfov 20 deg, 1280x720."""
    from tracer_b200 import harness as H
    return H.camera_rays((13, 2, 3), (0, 0, 0), np.float32(20 * np.pi / 180), 1280, 720)


def soup_rays_per_rank(name, world):
    return C5_FRAME_RAYS // world if name == "c5" else 8_000_000


def spawn_from_records(name, prim, recs, seed_base):
    """The timed batch of the Cornell workloads: bounce rays (c2bounce, c3) or shadow rays (c4) of the primary hits."""
    from tracer_b200 import harness as H
    if name == "c4":
        la, lb = H.scene_c4_lights(prim)
        return H.shadow_rays(recs, la, lb, seed_base)[0], True
    return H.bounce_rays(recs, seed_base)[0], False


def config_of(workload, prim, n, sort, flush, world):
    """Identical in the GPU arm and the reference arm (the driver compares the two dicts)."""
    return {"workload": WORKLOADS[workload], "query": "any-hit" if workload == "c4" else "closest-hit",
            "sharding": "ray batch per rank, scene replicated",
            "rays_per_step_per_gpu": int(n), "triangles": int(prim.nTri), "bvh_nodes": int(prim.bvhList.size),
            "ray_ordering": "TRQ_SORT_RAYS (origin cell x direction octant, inside the timed step)" if sort else "as given",
            "l2": ("flushed between steps (256 MB write)" if flush else
                   f"no flush: rays+hits stream {2 * n * 32 / 1e6:.0f} MB per step (> 126 MB L2)")}


class Work:
    """One workload on this rank: scene resident on the GPU, the ray batch, and `step()` = one pass of the hot path."""

    def __init__(self, name, D, rank, local_rank, world, sort_override=None):
        import torch
        from tracer_b200 import Scene, harness as H, layout as L, rays_to_torch
        self.name, self.device, self.world, self.rank = name, f"cuda:{local_rank}", world, rank
        t0 = time.time()
        prim = build_scene(name) if rank == 0 else None
        self.t_build = time.time() - t0
        self.prim = D.replicate_primitive(prim, src=0)
        self.scene = Scene(self.prim, local_rank)
        # TRQ_SORT_RAYS hint: only for the batch that is incoherent AND whose scene cannot live in L2 (C5)
        self.sort = (name == "c5") if sort_override is None else bool(sort_override)
        self.path = name in PATH_WORKLOADS
        self.any_hit, self.launches_per_step = name == "c4", 1
        dev = self.device
        if self.path:
            # device-resident wavefront (BASELINE configs[1]: "primary + 1 diffuse bounce"): castRay for every pixel,
            # trace, spawn the diffuse bounce of every hit (compacted, count stays on the device), trace that too.
            W, Hh = PATH_WORKLOADS[name]
            cam = ((278, 278, -800), (278, 278, 278), (0, 1, 0), np.float32(45 * (np.pi / 180)))
            self.W, self.Hh = W, Hh
            r0 = torch.empty((W * Hh, 8), dtype=torch.float32, device=dev); h0 = torch.empty_like(r0)
            r1 = torch.empty_like(r0); h1 = torch.empty_like(r0)
            s1 = torch.empty(W * Hh, dtype=torch.int32, device=dev); c1 = torch.zeros(1, dtype=torch.int64, device=dev)
            seed_base = rank << 32
            self.launches_per_step = 2
            self.h0, self.h1, self.r0, self.r1, self.s1 = h0, h1, r0, r1, s1
            scene = self.scene

            def step():
                scene.cast_rays(*cam, W, Hh, out=r0)
                scene.hit(r0, out=h0)
                scene.spawn_bounce(r0, h0, seed_base=seed_base, out=r1, src=s1, count=c1)
                scene.hit_indirect(r1, c1, out=h1)

            step(); torch.cuda.synchronize()
            self.n1 = int(c1.item())
            self.n = W * Hh + self.n1
            self.rays = np.concatenate([r0.cpu().numpy().view(L.ray_dtype).reshape(-1), r1[:self.n1].cpu().numpy().view(L.ray_dtype).reshape(-1)])
            self.step = step
            self.d_rays = None
        else:
            if name in ("c5", "soup1m"):
                n = soup_rays_per_rank(name, world)
                self.rays = H.random_rays(n, seed=2, first=rank * n)
            elif name == "c1":
                self.rays = c1_rays()
            else:
                W, Hh = (1920, 1080) if name == "c2bounce" else (3840, 2160)
                d = rays_to_torch(H.cornell_camera_rays(W, Hh), dev)
                recs = self.scene.expand(d, self.scene.hit(d)).cpu().numpy().view(L.record_dtype).reshape(-1)
                del d
                self.rays, _ = spawn_from_records(name, self.prim, recs, rank << 32)
            self.n = self.rays.size
            self.d_rays = rays_to_torch(self.rays, dev)
            self.d_hits = torch.empty((self.n, 8), dtype=torch.float32, device=dev)
            scene, d_rays, d_hits, any_hit, sort = self.scene, self.d_rays, self.d_hits, self.any_hit, self.sort

            def step():
                scene.hit(d_rays, any=any_hit, out=d_hits, sort=sort)
            self.step = step
            # the same batch WITHOUT the TRQ_SORT_RAYS hint: on a tree much larger than L2 the library examines the batch itself
            self.step_unhinted = lambda: scene.hit(d_rays, any=any_hit, out=d_hits, sort=None)

    def hits(self):
        """Device hit records of the last step (wavefronts: primary wave, then the bounce wave)."""
        import torch
        if self.path:
            return torch.cat([self.h0, self.h1[:self.n1]])
        return self.d_hits

    def snapshot(self):
        """(rays, hits) of the LAST step, index-aligned. For the device-resident wavefronts the bounce wave is compacted
        with one atomic per warp, so its ORDER differs from step to step: rays and hits are read back together."""
        import torch
        from tracer_b200 import layout as L
        if self.path:
            rays = torch.cat([self.r0, self.r1[:self.n1]]).cpu().numpy().view(L.ray_dtype).reshape(-1)
            return rays, self.hits()
        return self.rays, self.d_hits

    def close(self):
        self.scene.close()
        self.d_rays = self.d_hits = self.h0 = self.h1 = self.r0 = self.r1 = self.s1 = None


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock and clock-event (throttle) reasons sampled IN PROCESS through NVML from a background thread, about once
    per millisecond, from before the warm-up until after the timed region; samples whose timestamp falls inside a marked
    window are reported. Falls back to `nvidia-smi -lms 20` when NVML cannot be loaded."""
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"),
               (0x80, "hw_power_brake_slowdown"))

    def __init__(self, cuda_index):
        self.rows, self.windows, self._stop = [], [], False
        self.nvml = self.handle = self.proc = self.thread = None
        self.source = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                uuid = str(torch.cuda.get_device_properties(cuda_index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(cuda_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml, self.source = pynvml, "nvml (in-process thread, ~1 ms period)"
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
        except Exception:
            self.nvml = None
            self._start_smi(cuda_index)

    def _poll(self):
        nv, h = self.nvml, self.handle
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop:
            try:
                self.rows.append((time.time(), float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), int(get_reasons(h))))
            except Exception:
                pass
            time.sleep(0.0005)

    def _start_smi(self, idx):
        fields = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                  "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        self.path = tempfile.mktemp(prefix="trq_clocks_", suffix=".csv")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(idx), f"--query-gpu={fields}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            self.source = "nvidia-smi -lms 20"
        except OSError:
            self.proc = None

    def mark(self, name, t0, t1):
        self.windows.append((name, t0, t1))

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "window": None, "source": self.source}
        self._stop = True
        rows = []
        if self.thread is not None:
            self.thread.join(timeout=2)
            rows = [(t, mhz, [name for bit, name in self.REASONS if r & bit]) for t, mhz, r in self.rows]
            out["sm_max_mhz"] = self.max_mhz
        elif self.proc is not None:
            import datetime
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
            names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
            try:
                for line in open(self.path):
                    p = [x.strip() for x in line.split(",")]
                    if len(p) < 7:
                        continue
                    try:
                        ts = datetime.datetime.strptime(p[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                        rows.append((ts, float(p[1]), [n for n, v in zip(names, p[3:7]) if v.lower().startswith("active")]))
                        out["sm_max_mhz"] = float(p[2])
                    except ValueError:
                        continue
                os.unlink(self.path)
            except OSError:
                pass
        for name, lo, hi in self.windows:                         # first window with enough samples wins
            sel = [r for r in rows if lo <= r[0] <= hi]
            if len(sel) >= 3:
                out.update({"sm_mhz": float(np.median([r[1] for r in sel])), "reasons": sorted({n for r in sel for n in r[2]}),
                            "samples": len(sel), "window": name})
                break
        return out


# ----------------------------------------------------------------------------------------------- measurement
def time_steps(D, step, steps, flush=None):
    """K steps between barrier + synchronize, CUDA events on the current stream; returns (ms, wall t0, wall t1)."""
    import torch
    D.barrier(); torch.cuda.synchronize()
    t0 = time.time()
    if flush is None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
    else:
        evs = []
        for _ in range(steps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); step(); e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        ms = sum(x.elapsed_time(y) for x, y in evs)
    t1 = time.time()
    D.barrier()
    return ms, t0, t1


def measure(D, work, steps, warmup, flush=None, sampler=None):
    from tracer_b200 import launch_count
    import torch
    for _ in range(max(warmup, 3)):
        work.step()
    torch.cuda.synchronize()
    work.scene.profile(True)
    l0 = launch_count()
    ms, t0, t1 = time_steps(D, work.step, steps, flush)
    launches = launch_count() - l0
    nl, trace_ms, _ = work.scene.profile_read()
    work.scene.profile(False)
    if sampler is not None:
        sampler.mark("timed region", t0, t1)
    total_ms = D.max_over_ranks(ms)
    total_rays = D.sum_over_ranks(work.n)
    return {"total_ms": total_ms, "total_rays": total_rays, "value": total_rays * steps / total_ms / 1e3,
            "ms_per_step": total_ms / steps, "launches": int(launches),
            "kernel_ms": trace_ms / max(1, nl) * work.launches_per_step}


def measure_unhinted(D, work, steps):
    """C5 without the caller's hint: the library's own coherence check decides (three extra launches per step inside the timed region)."""
    import torch
    for _ in range(3):
        work.step_unhinted()
    torch.cuda.synchronize()
    ms, _, _ = time_steps(D, work.step_unhinted, steps)
    total_ms = D.max_over_ranks(ms)
    return {"value": round(D.sum_over_ranks(work.n) * steps / total_ms / 1e3, 2), "unit": UNIT, "steps": steps,
            "ms_per_step": round(total_ms / steps, 4),
            "how": "no TRQ_SORT_RAYS flag: a probe over 64 K sampled rays measures how many neighbouring rays share (cell, octant); the queue is ordered when fewer than half do"}


def bytes_per_ray(work, nthreads):
    """Algorithmic bytes per ray from the instrumented oracle's step counters on a strided pilot of the batch."""
    from oracle.pyoracle import Port
    pilot = work.rays[:: max(1, work.n // 40000)]
    tot = Port().trace(work.prim, pilot, any=work.any_hit, nthreads=nthreads)["totals"]
    return tot["bytes"] / max(1, tot["n_rays"])


def parity_on(work, idx, nthreads):
    """GPU records of the last step at ray indices `idx` against the oracle on the same rays."""
    import torch
    from oracle.pyoracle import Port
    from tracer_b200 import layout as L
    rays, hits = work.snapshot()
    sub = np.ascontiguousarray(rays[idx])
    want = Port().trace(work.prim, sub, any=work.any_hit, nthreads=nthreads)["hits"]
    got = hits[torch.from_numpy(np.asarray(idx, dtype=np.int64)).to(work.device)].cpu().numpy().view(L.hit_dtype).reshape(-1)
    ids_ok = all(np.array_equal(got[k], want[k]) for k in ("flags", "pType", "pIndex", "leafNode"))
    t_ok = np.array_equal(got["t"].view(np.uint32), want["t"].view(np.uint32))
    tri = want["pType"] == 3                                  # barycentrics: bit-exact for triangle hits
    uv_ok = all(np.array_equal(got[k][tri].view(np.uint32), want[k][tri].view(np.uint32)) for k in ("u", "v"))
    return {"rays": int(sub.size), "ids_bit_exact": bool(ids_ok), "t_bit_exact": bool(t_ok), "barycentrics_bit_exact": bool(uv_ok)}


def dump_outputs(work, out_dir):
    """--dump-outputs: what the last timed step returned to its caller, as DIR/<struct>_<field>.npy, one file per field of
    the C-ABI structs (trq_hit; for the wavefronts also the trq_ray batches they produce). Float fields are written as
    float32, integer fields as float64 (exact). Row i of every file belongs to the ray at position ray_index[i] of the
    step's batch. A batch too large for DUMP_BYTES is sampled with a fixed seed, so runs with the same arguments write
    the same rays. The wavefronts compact their bounce wave in a different order every step, so that wave is written in
    source-pixel order."""
    import torch
    from tracer_b200 import layout as L
    if work.path:
        order = torch.argsort(work.s1[:work.n1])
        out = {"ray": (L.ray_dtype, torch.cat([work.r0, work.r1[:work.n1][order]])),
               "hit": (L.hit_dtype, torch.cat([work.h0, work.h1[:work.n1][order]]))}
    else:
        out = {"hit": (L.hit_dtype, work.d_hits)}

    def as_float(a):
        return a.astype(np.float32 if a.dtype.kind == "f" else np.float64)

    per_ray = 8 + sum(as_float(np.zeros(1, dt)[f]).nbytes for dt, _ in out.values() for f in dt.names)
    n = work.n
    m = min(n, DUMP_BYTES // per_ray)
    idx = np.arange(n) if m == n else np.sort(np.random.default_rng(0).choice(n, m, replace=False))
    sel = torch.from_numpy(idx).to(work.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, (dt, rows) in out.items():
        rec = rows[sel].cpu().numpy().view(dt).reshape(-1)
        for f in dt.names:
            np.save(os.path.join(out_dir, f"{name}_{f}.npy"), as_float(rec[f]))
    np.save(os.path.join(out_dir, "ray_index.npy"), idx.astype(np.float64))


def roofline_of(name, bpr, n, kernel_ms, step_ms, launches_per_step, hbm_peak, peak_src, l2_gbs, prof):
    """achieved = algorithmic bytes per launch / kernel time; peak = the ceiling of the level that bounds the workload.
    prof: this workload's entry of profiles/traffic.json (ncu --set full capture of the same launch), or None."""
    bound = BOUND[name]
    traffic = None if not prof else prof.get("traffic_gb")
    if traffic is not None and prof.get("rays_per_launch") and prof["rays_per_launch"] != n // launches_per_step:
        traffic = round(traffic * (n / launches_per_step) / prof["rays_per_launch"], 4)     # captured at another shard size: scaled per ray
    achieved = bpr * n / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else None
    if bound == "l2" and l2_gbs:
        peak, src = l2_gbs, "L2 read bandwidth measured on this GPU in this run (trq_probe_bandwidth: 16-byte loads over a 32 MB set, all SMs); MEASURED_PEAKS.json has no L2 figure"
    else:
        peak, src = hbm_peak, peak_src
    r = {"bound": bound, "kernel": "trace_packed_kernel", "achieved": None if achieved is None else round(achieved, 1),
         "peak": round(peak, 1), "unit": "GB/s", "frac": None if achieved is None else round(achieved / peak, 4),
         "traffic": traffic, "traffic_unit": "GB per launch (ncu dram__bytes_read+write)", "peak_source": src,
         "algorithmic_bytes_per_ray": round(bpr, 1), "algorithmic_gb_per_launch": round(bpr * n / launches_per_step / 1e9, 3),
         "kernel_ms": round(kernel_ms, 4), "trace_launches_per_step": launches_per_step,
         "kernel_share_of_step": round(kernel_ms / max(1e-9, step_ms), 4),
         "hbm_peak": hbm_peak, "frac_of_hbm_peak": None if achieved is None else round(achieved / hbm_peak, 4),
         # what actually crosses the DRAM pins (ncu, per launch) as a fraction of the HBM peak over the kernel's live duration
         "dram_frac": None if (traffic is None or kernel_ms <= 0) else round(traffic * launches_per_step / (kernel_ms * 1e-3) / hbm_peak, 4),
         "l2_read_peak_gbs_measured": None if not l2_gbs else round(l2_gbs, 1)}
    if prof:      # what ncu says bounds the kernel: the L1 data pipe (one wavefront per divergent 32-byte lane request)
        r["ncu"] = {k: prof[k] for k in ("l1tex_pct", "lanes_per_inst", "issue_active_pct", "l1_hit_pct", "l2_hit_pct", "dram_pct_of_peak") if k in prof}
    return r


# ----------------------------------------------------------------------------------------------- CPU reference
def cpu_reference(prim, rays, any_hit, budget_s, nthreads):
    """Time the reference's Scene::hit (verbatim build if present, else the C port) on `rays` subsampled so that one
    pass takes about budget_s. Returns (Mrays/s, kind, cores, sample description, stride)."""
    from oracle.pyoracle import Port, Reference
    port = Port()
    use_ref = Reference.available()
    ref = Reference() if use_ref else None

    def run(sub):
        t = time.perf_counter()
        if use_ref:
            ref.trace_lite(prim, sub, any=any_hit, nthreads=nthreads)
        else:
            port.trace(prim, sub, any=any_hit, nthreads=nthreads)
        return time.perf_counter() - t

    pilot = rays[:: max(1, rays.size // 40000)]
    run(pilot[: max(1, pilot.size // 4)])                       # page in
    dt = run(pilot)
    rate = pilot.size / max(dt, 1e-6)
    want = int(min(rays.size, max(pilot.size, rate * budget_s)))
    stride = max(1, rays.size // want)
    sub = np.ascontiguousarray(rays[::stride])
    passes, dt = 0, 0.0
    while passes < 12 and (passes == 0 or dt < 0.8 * budget_s):        # ~budget_s of CPU work even when one pass is short
        dt += run(sub)
        passes += 1
    kind = "reference" if use_ref else "port"
    sample = ("every ray of the batch" if stride == 1 else f"every {stride}th ray of the batch") + \
             f" ({sub.size} rays) x {passes} passes, {dt:.1f} s of CPU work"
    return sub.size * passes / dt / 1e6, kind, nthreads, sample, stride


# ----------------------------------------------------------------------------------------------- arms
def run_reference_arm(a):
    rank, _, world = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("LOCAL_RANK", "0"), ("WORLD_SIZE", "1")))
    if rank != 0:
        return 0
    from oracle.pyoracle import Port, Reference
    from tracer_b200 import harness as H
    name = a.workload
    prim = build_scene(name)
    nthreads = os.cpu_count() or 1
    use_ref = Reference.available()
    eng = Reference() if use_ref else Port()
    rec_fn = (lambda r: eng.trace(prim, r, nthreads=nthreads)) if use_ref else (lambda r: eng.trace(prim, r, records=True, nthreads=nthreads)["records"])
    # the SAME batch as the GPU arm's rank 0 (generated without a GPU: the primary hits come from the CPU reference),
    # so that both arms describe one config; the timed steps then run on a strided sample of it
    any_hit = name == "c4"
    if name in ("c5", "soup1m"):
        n_full = soup_rays_per_rank(name, max(1, a.gpus))
        rays = H.random_rays(n_full // 16, seed=2)               # a prefix of rank 0's shard: same distribution, bounded memory
        pre = 16
    elif name == "c1":
        rays, n_full, pre = c1_rays(), 1280 * 720, 1
    else:
        W, Hh = (1920, 1080) if name in ("c2", "c2bounce") else (3840, 2160)
        primary = H.cornell_camera_rays(W, Hh)
        recs = rec_fn(primary)
        spawned, any_hit = spawn_from_records(name, prim, recs, 0)
        if name in PATH_WORKLOADS:                               # both waves of the wavefront
            rays = np.concatenate([primary, spawned])
        else:
            rays = spawned
        n_full, pre = rays.size, 1

    def run(sub):
        t = time.perf_counter()
        if use_ref:
            eng.trace_lite(prim, sub, any=any_hit, nthreads=nthreads)
        else:
            eng.trace(prim, sub, any=any_hit, nthreads=nthreads)
        return time.perf_counter() - t

    pilot = rays[:: max(1, rays.size // 20000)]
    rate = pilot.size / max(run(pilot), 1e-6)
    budget = min(3.0, 120.0 / max(1, a.steps + a.warmup))
    stride = max(1, int(rays.size / max(pilot.size, rate * budget)))
    sub = np.ascontiguousarray(rays[::stride])
    for _ in range(a.warmup):
        run(sub)
    t = sum(run(sub) for _ in range(a.steps))
    v = sub.size * a.steps / t / 1e6
    kind = "reference" if use_ref else "port"
    sample = f"{sub.size} rays per step: every {pre * stride}th ray of the {n_full}-ray batch"
    sort = name == "c5"
    line = {
        "impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": round(t / a.steps * 1e3, 3), "higher_is_better": True,
        "scaling": "strong" if name == "c5" else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(name, prim, n_full, sort, a.flush_l2, max(1, a.gpus)),
        "cpu_baseline": {"value": round(v, 4), "unit": UNIT, "cores": nthreads, "kind": kind, "sample": sample},
        "e2e": {"value": round(v, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def measure_gather(D, work, steps, rank, world):
    """Every rank's hit records delivered to every rank: trq_trace_gather (tiles of finished records shipped to every peer
    over NVLink while the traversal runs), trq_hit and trq_hit16 records, and NCCL's all-gather beside it.
    A figure whose records do not check out is nulled."""
    import torch
    n_common = int(-D.max_over_ranks(-float(work.n)))                      # ranks trace slightly different batch sizes
    g_rays = work.d_rays[:n_common].contiguous()
    any_hit, sort, scene, device = work.any_hit, work.sort, work.scene, work.device
    out = {"unit": UNIT, "steps": steps, "rays_per_rank": n_common}
    # local truth: this rank's own records, 32-byte and 16-byte form
    own32 = scene.hit(g_rays, any=any_hit, sort=sort).clone()
    own16 = scene.hit(g_rays, any=any_hit, sort=sort, hit16=True).clone()
    m = min(n_common, 1 << 18)
    ref32 = D.gather_hits(own32[:m].contiguous())                           # NCCL gather of a slice: what slot r must hold
    ref16 = [t[:, :4].contiguous() for t in D.gather_hits(torch.cat([own16[:m], torch.zeros_like(own16[:m])], dim=1))]

    # ---- NCCL: trace chunk by chunk, all-gather each chunk on a second stream under the tracing of the next
    g_local = torch.empty((n_common, 8), dtype=torch.float32, device=device)
    g_all = torch.empty((world, n_common, 8), dtype=torch.float32, device=device)
    for _ in range(3):
        D.trace_and_gather(scene, g_rays, g_local, g_all, any=any_hit, sort=sort)
    ms, _, _ = time_steps(D, lambda: D.trace_and_gather(scene, g_rays, g_local, g_all, any=any_hit, sort=sort), steps)
    g_ms = D.max_over_ranks(ms)
    ok = bool(torch.equal(g_all[rank].view(torch.int32), own32.view(torch.int32)))
    ok = bool(-D.max_over_ranks(-float(ok)) == 1.0)
    out["nccl_overlapped"] = {"value": round(n_common * world * steps / g_ms / 1e3, 2) if ok else None, "ms_per_step": round(g_ms / steps, 4),
                              "chunks": 4, "own_shard_matches": ok, "how": "dist.trace_and_gather: NCCL all-gather per chunk on a second stream"}
    del g_all, g_local

    # ---- fused: the traversal kernel itself stores every record to every rank
    try:
        hg = D.HitGather(scene, n_common)
    except RuntimeError as e:                                 # raised on every rank alike (HitGather agrees on failures)
        out["peer_gather_error"] = str(e)
        return out
    for h16, key, own, ref in ((False, "trq_hit", own32, ref32), (True, "trq_hit16", own16, ref16)):
        for _ in range(3):
            hg.trace(g_rays, any=any_hit, sort=sort, hit16=h16); hg.wait()
        res = {}

        def gstep():
            hg.trace(g_rays, any=any_hit, sort=sort, hit16=h16)
            res["all"], res["counts"] = hg.wait()
        ms, _, _ = time_steps(D, gstep, steps)
        published = True
        try:
            hg.status()
        except RuntimeError:                                  # a peer never published: reported, and no rank leaves the collectives below
            published = False
        p_ms = D.max_over_ranks(ms)
        p_all, p_counts = res["all"], res["counts"]
        full = published and bool((p_counts == n_common).all())
        full = full and bool(torch.equal(p_all[rank].contiguous().view(torch.int32), own.view(torch.int32)))
        full = full and all(bool(torch.equal(p_all[r, :m].contiguous().view(torch.int32), ref[r].view(torch.int32))) for r in range(world))
        full = bool(-D.max_over_ranks(-float(full)) == 1.0)
        rec = 16 if h16 else 32
        out[key] = {"value": round(n_common * world * steps / p_ms / 1e3, 2) if full else None, "ms_per_step": round(p_ms / steps, 4),
                    "record_bytes": rec, "peer_store_bytes_per_rank_per_step": int(n_common * (world - 1) * rec),
                    "nvlink_egress_gbs_per_gpu": round(n_common * (world - 1) * rec / (p_ms / steps * 1e-3) / 1e9, 1),
                    "all_slots_match": full}
    hg.close()
    out["value"] = out["trq_hit"]["value"]
    out["ms_per_step"] = out["trq_hit"]["ms_per_step"]
    out["all_slots_match"] = out["trq_hit"]["all_slots_match"] and out["trq_hit16"]["all_slots_match"]
    out["how"] = ("trq_trace_gather: the trace kernel counts finished records per 2048-record tile; a TMA sender kernel sharing the SMs "
                  "with it (one thread per SM, cp.async.bulk through 2 x 12 KB of shared memory) ships each complete tile to every rank's "
                  "buffer over NVLink peer memory, under the traversal, and publishes (count, step)")
    return out


def run_gpu_arm(a):
    # stdout carries exactly ONE line (the JSON); anything libraries print there (e.g. "NCCL version ...") goes to stderr
    json_fd = os.dup(1)
    os.dup2(2, 1)
    import torch

    from tracer_b200 import dist as D, probe_bandwidth
    rank, local_rank, world = D.init()
    if world != a.gpus:
        log(f"warning: --gpus {a.gpus} but WORLD_SIZE={world}")
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    device = f"cuda:{local_rank}"
    nthreads = os.cpu_count() or 1
    t_start = time.time()

    sampler = ClockSampler(local_rank)                  # runs from before the warm-up to the end of the last timed region
    work = Work(a.workload, D, rank, local_rank, world, a.sort)
    scene, n, any_hit, sort, path = work.scene, work.n, work.any_hit, work.sort, work.path
    if rank == 0:
        log(f"# scene {scene.info}, build {work.t_build:.1f}s, {n} rays/step/rank")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device) if a.flush_l2 else None

    # ---- timed region: K steps, device events, barrier + synchronize on both sides
    m = measure(D, work, a.steps, a.warmup, flush, sampler)
    value, total_ms, total_rays = m["value"], m["total_ms"], m["total_rays"]
    if a.dump_outputs and rank == 0:
        dump_outputs(work, a.dump_outputs)
    unhinted = measure_unhinted(D, work, a.steps) if a.workload == "c5" and sort else None
    hit_frac = float((work.hits()[:, 7].view(torch.int32) & 1).float().mean())
    d_hits_ref = work.hits().clone()

    # ---- e2e: host (pinned) rays in, host hits out, through the C-ABI host-pointer path
    h_hits = torch.empty((n, 8), dtype=torch.float32).pin_memory()
    e2e_steps = a.steps
    e2e_extra = {}
    if path:
        W, Hh, n1 = work.W, work.Hh, work.n1
        # inputs are the camera (52 bytes); both hit buffers come back to pinned host memory every step

        def e2e_step():
            work.step()
            h_hits[: W * Hh].copy_(work.h0, non_blocking=True)
            h_hits[W * Hh:].copy_(work.h1[:n1], non_blocking=True)
            torch.cuda.synchronize()
        h2d_bytes, d2h_bytes = 52, int(n * 32)
    else:
        h_rays = torch.from_numpy(work.rays.view(np.float32).reshape(-1, 8)).pin_memory()

        def e2e_step():
            scene.hit_host(h_rays.data_ptr(), n, h_hits.data_ptr(), any=any_hit, sort=sort)
        h2d_bytes, d2h_bytes = int(n * 32), int(n * 32)

    def wall(fn, k):
        for _ in range(2):
            fn()
        D.barrier(); torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(k):
            fn()
        torch.cuda.synchronize()
        return D.max_over_ranks(time.perf_counter() - t)

    e2e_s = wall(e2e_step, e2e_steps)
    e2e_value = total_rays * e2e_steps / e2e_s / 1e6
    # the host path must produce the same bytes as the device path (wavefronts: the records of that very step)
    # (compared as bit patterns: sphere uv can be NaN -- asinf just outside [-1, 1] -- and NaN != NaN as floats)
    same = bool(torch.equal(h_hits.view(torch.int32), (work.hits() if path else d_hits_ref).cpu().view(torch.int32)))
    if not path:
        # the opt-in 16-byte record: half the D2H bytes
        h_hits16 = torch.empty((n, 4), dtype=torch.float32).pin_memory()
        s16 = wall(lambda: scene.hit_host(h_rays.data_ptr(), n, h_hits16.data_ptr(), any=any_hit, sort=sort, hit16=True), e2e_steps)
        from tracer_b200 import layout as L
        want16 = L.pack_hit16(d_hits_ref.cpu().numpy().view(L.hit_dtype).reshape(-1))
        e2e_extra["e2e_hit16"] = {"value": round(total_rays * e2e_steps / s16 / 1e6, 2), "unit": UNIT, "h2d_bytes_per_step": int(n * 32),
                                  "d2h_bytes_per_step": int(n * 16), "steps": e2e_steps,
                                  "equals_packed_device_records": bool(np.array_equal(h_hits16.numpy().view(np.uint8).reshape(-1), want16.view(np.uint8).reshape(-1)))}
        if a.workload == "c5" and sort:
            # the same host-pointer call WITHOUT the caller's ordering hint (the library examines each 1 M-ray chunk itself)
            su = wall(lambda: scene.hit_host(h_rays.data_ptr(), n, h_hits.data_ptr(), any=any_hit, sort=False), e2e_steps)
            e2e_extra["e2e_unhinted"] = {"value": round(total_rays * e2e_steps / su / 1e6, 2), "unit": UNIT, "steps": e2e_steps,
                                         "equals_device_path": bool(torch.equal(h_hits.view(torch.int32), d_hits_ref.cpu().view(torch.int32)))}
        # same traffic as e2e, but the K calls are queued back to back (TRQ_HOST_ASYNC, two alternating pinned result
        # buffers) so that one call's D2H overlaps the next call's H2D; collected once at the end
        h_hits2 = torch.empty((n, 8), dtype=torch.float32).pin_memory()
        outs = (h_hits, h_hits2)
        for k in range(2):
            scene.hit_host(h_rays.data_ptr(), n, outs[k].data_ptr(), any=any_hit, sort=sort, asynchronous=True)
        scene.host_sync()
        D.barrier(); torch.cuda.synchronize()
        t = time.perf_counter()
        for k in range(e2e_steps):
            scene.hit_host(h_rays.data_ptr(), n, outs[k & 1].data_ptr(), any=any_hit, sort=sort, asynchronous=True)
        scene.host_sync()
        pipe_s = D.max_over_ranks(time.perf_counter() - t)
        e2e_extra["e2e_pipelined"] = {"value": round(total_rays * e2e_steps / pipe_s / 1e6, 2), "unit": UNIT, "steps": e2e_steps,
                                      "note": "K TRQ_HOST_ASYNC calls queued back to back + one trq_host_sync; same bytes per step as e2e",
                                      "equals_device_path": bool(torch.equal(h_hits2.view(torch.int32), d_hits_ref.cpu().view(torch.int32)))}
        del h_hits2, h_hits16
    del h_hits

    # ---- multi-GPU, second figure (SURVEY 8d "with and without hit all-gather")
    with_gather = None
    if world > 1 and not path:
        with_gather = measure_gather(D, work, a.steps, rank, world)

    # ---- multi-GPU: scene checksum agreement + gathered hit count (not timed)
    gathered = None
    if world > 1:
        cs = D.checksum_primitive(work.prim)
        lo, hi = D.max_over_ranks(float(cs % (1 << 52))), -D.max_over_ranks(-float(cs % (1 << 52)))
        assert lo == hi, "scene broadcast checksum differs across ranks"
        parts = D.gather_hits(d_hits_ref[: min(n, 1 << 20)])
        gathered = int(sum(p.shape[0] for p in parts))

    # ---- the memory system as measured on this GPU right now (L2 has no entry in MEASURED_PEAKS.json)
    hbm_peak, peak_src = peaks()
    try:
        l2_gbs, hbm_read_gbs = probe_bandwidth(local_rank, "l2"), probe_bandwidth(local_rank, "hbm")
    except Exception as e:
        log(f"# bandwidth probe failed: {e!r}")
        l2_gbs = hbm_read_gbs = None
    traffic = traffic_table()

    # ---- CPU baseline + algorithmic bytes + parity (rank 0; the timed baseline at N=1 only)
    bpr, cpu, parity_ok = BYTES_PER_RAY_FALLBACK[a.workload], None, None
    if rank == 0:
        try:
            work.step(); torch.cuda.synchronize()                 # work.hits() = the records of this batch again
            bpr = bytes_per_ray(work, nthreads)
            if world == 1 and not a.no_cpu_baseline:
                v, kind, cores, sample, stride = cpu_reference(work.prim, work.rays, any_hit, a.cpu_budget, nthreads)
                cpu = {"value": round(v, 4), "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}
                # parity on the timed sample: GPU records of those rays vs the oracle (for C3: every ray of the batch)
                cpu["parity_on_sample"] = parity_on(work, np.arange(0, n, stride), cores)
                parity_ok = all(v for k, v in cpu["parity_on_sample"].items() if k != "rays")
                if a.workload == "c1":
                    # the config's NAMED baseline: RT_Nextweek's own CPU BVH (restated in C, oracle/nextweek_bvh.c; parity unpinned)
                    from oracle.pyoracle import Nextweek
                    from tracer_b200 import layout as L
                    nw = Nextweek(work.prim.sphereList)
                    nw.trace(work.rays[:50000], nthreads=cores)
                    t0 = time.perf_counter(); ids, _ = nw.trace(work.rays, nthreads=cores); dt = time.perf_counter() - t0
                    mine = work.hits().cpu().numpy().view(L.hit_dtype).reshape(-1)
                    hit = (mine["flags"] & 1) == 1
                    cpu["nextweek_bvh"] = {"value": round(n / dt / 1e6, 4), "unit": UNIT, "cores": cores, "kind": "port",
                                           "sample": f"all {n} rays, {dt:.1f} s",
                                           "same_sphere_as_gpu": round(float(np.mean(ids[hit] == mine["pIndex"][hit])), 6)}
        except Exception as e:  # the oracle is test infrastructure: never let it take the GPU numbers down
            log(f"# cpu baseline unavailable: {e!r}")
    main_roof = roofline_of(a.workload, bpr, n, m["kernel_ms"], m["ms_per_step"], work.launches_per_step, hbm_peak, peak_src, l2_gbs,
                            traffic.get(a.workload + ("_sorted" if sort and a.workload + "_sorted" in traffic else "")))
    main_cfg = config_of(a.workload, work.prim, n, sort, a.flush_l2, world)
    kernel_cfg = scene.kernel_config()
    work.close()
    del d_hits_ref
    torch.cuda.empty_cache()

    # ---- BASELINE.json's other configs, each: K steps device-resident, kernel time, roofline, parity on a sample
    extras = None
    if a.workload == "c3" and not a.no_extra and not a.flush_l2:
        extras = {}
        for wname in EXTRA_WORKLOADS:
            if time.time() - t_start > a.extra_deadline:
                extras[wname] = {"skipped": f"run already at {time.time() - t_start:.0f} s"}
                continue
            try:
                w = Work(wname, D, rank, local_rank, world)
                r = measure(D, w, a.steps, a.warmup)
                e = {"config": WORKLOADS[wname], "query": "any-hit" if w.any_hit else "closest-hit", "value": round(r["value"], 2), "unit": UNIT,
                     "steps": a.steps, "ms_per_step": round(r["ms_per_step"], 4), "rays_per_step_per_gpu": int(w.n),
                     "scaling": "strong" if wname == "c5" else "weak", "gpu_launches": r["launches"],
                     "ray_ordering": "TRQ_SORT_RAYS" if w.sort else "as given", "kernel_config": w.scene.kernel_config()}
                if rank == 0:
                    try:
                        wb = bytes_per_ray(w, nthreads)
                        idx = np.arange(0, w.n, max(1, w.n // 100_000))
                        e["parity_on_sample"] = parity_on(w, idx, nthreads)
                    except Exception as ex:
                        wb = BYTES_PER_RAY_FALLBACK[wname]
                        log(f"# {wname}: oracle unavailable: {ex!r}")
                    e["roofline"] = roofline_of(wname, wb, w.n, r["kernel_ms"], r["ms_per_step"], w.launches_per_step, hbm_peak, peak_src, l2_gbs,
                                                traffic.get(wname + "_sorted" if w.sort and wname + "_sorted" in traffic else wname))
                if wname == "c5":
                    e["unhinted"] = measure_unhinted(D, w, a.steps)
                extras[wname] = e
                w.close()
                del w
                torch.cuda.empty_cache()
            except Exception as ex:
                extras[wname] = {"error": repr(ex)[:200]}
                log(f"# workload {wname} failed: {ex!r}")
    clocks = sampler.stop()

    if rank != 0:
        D.barrier()
        _shutdown()
        return 0

    line = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": round(m["ms_per_step"], 4), "higher_is_better": True, "scaling": "strong" if a.workload == "c5" else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": main_cfg, "hit_fraction": round(hit_frac, 4), "kernel_config": kernel_cfg,
        "roofline": main_roof,
        "cpu_baseline": cpu,
        "e2e": {"value": round(e2e_value, 2), "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "steps": e2e_steps, "host_path_equals_device_path": same, "timing": "wall clock around K synchronous C-ABI calls, max over ranks"},
        "gpu_launches": m["launches"],
        "clocks": clocks,
    }
    if unhinted is not None:
        line["unhinted"] = unhinted
    line.update(e2e_extra)
    if gathered is not None:
        line["gathered_hits_checked"] = gathered
    if with_gather is not None:
        line["with_hit_allgather"] = with_gather
    if extras is not None:
        line["workloads"] = extras
    sys.stdout.flush()
    os.write(json_fd, (json.dumps(line) + "\n").encode())
    D.barrier()
    _shutdown()
    # a fast kernel whose results differ from the reference's is not done: the line is printed, the exit code says so
    if parity_ok is False or not same:
        log("# PARITY FAILURE: see cpu_baseline.parity_on_sample / e2e.host_path_equals_device_path")
        return 2
    return 0


def _shutdown():
    import torch.distributed as dist
    if dist.is_initialized():
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--flush-l2", action="store_true")
    ap.add_argument("--sort", type=int, default=None, help="force the TRQ_SORT_RAYS hint on (1) / off (0); default: on for c5 only")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip BASELINE.json's other configs (workloads: c1, c2, c4, c5)")
    ap.add_argument("--extra-deadline", type=float, default=240.0, help="do not start another extra workload after this many seconds")
    ap.add_argument("--cpu-budget", type=float, default=10.0, help="seconds of CPU work for the cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the records of the last timed step (rank 0) as DIR/*.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.impl == "reference" and a.dump_outputs:
        ap.error("--dump-outputs writes the GPU path's records; the reference arm has none to write")
    if a.impl == "reference":
        return run_reference_arm(a)
    return run_gpu_arm(a)


if __name__ == "__main__":
    sys.exit(main())
