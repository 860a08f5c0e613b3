#!/usr/bin/env python
"""Developer tool: the Morton-order builder against the SAH builder -- build and rebuild times, and what each tree costs
the traversal.
Usage: python tools/morton_perf.py [out.txt]      (prints the report; also writes it to out.txt when given)

On C3 (1.0 M triangles) and a 1 M-triangle soup:
  1. device tree build, trq_bvh_build_tree_device against trq_bvh_build_tree_morton_device (CUDA events around the
     synchronous call; the leaves are copied back in before each build, outside the events);
  2. trq_scene_rebuild without and with TRQ_BUILD_MORTON (host clock around the synchronous call);
  3. closest-hit Mrays/s on each tree (CUDA events): C3's diffuse bounce rays from 3840x2160 primary hits, 4 M random rays
     through the soup; the hits of both trees checked against port.trace on a sample of 20,000 rays;
  4. each tree's maxDepth;
  5. one Morton rebuild of C3 under torch.profiler: time per kernel (a separate pass; the profiler slows the host).
Every timed call is warmed up first; every time is the median of the repetitions."""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from tracer_b200 import DevicePrimitive, Scene, harness as H, layout as L, rays_to_torch  # noqa: E402
from tracer_b200._lib import check, lib  # noqa: E402

REPS = 20
SAMPLE = 20_000
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()


def median_ms(fn, reps=REPS, events=False, before=None):
    if before:
        before()
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        if before:
            before()
        torch.cuda.synchronize()
        if events:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); b.synchronize()
            out.append(a.elapsed_time(b))
        else:
            t = time.perf_counter(); fn(); torch.cuda.synchronize()
            out.append(1e3 * (time.perf_counter() - t))
    return float(np.median(out))


def device_build_ms(leaves_dev, n, fn):
    buf = torch.empty((2 * n - 1) * 64, dtype=torch.uint8, device="cuda")
    nn, depth = C.c_uint32(0), C.c_uint32(0)

    def reset():
        buf[: n * 64].copy_(leaves_dev)

    ms = median_ms(lambda: check(fn(buf.data_ptr(), n, 0, C.byref(nn), C.byref(depth)), fn.__name__), events=True, before=reset)
    return ms, depth.value


def oracle_check(port, prim, rays, hits, where):
    pick = np.random.default_rng(1).choice(rays.size, min(SAMPLE, rays.size), replace=False)
    want = port.trace(prim, rays[pick], nthreads=os.cpu_count() or 8)["hits"]
    got = hits[pick]
    for k in ("t", "pType", "pIndex", "leafNode", "u", "v", "flags"):
        assert np.array_equal(got[k].view(np.uint32), want[k].view(np.uint32)), f"{where}: {k} differs from the oracle"
    return pick.size


def compare(name, prim, rays_np, port):
    n = prim.nTri
    say(f"--- {name}: {n} triangles, {rays_np.size} rays")
    leaves = prim.bvhList[1:n + 1].copy()
    leaves_dev = dev(leaves)
    t_sah, d_sah = device_build_ms(leaves_dev, n, lib.trq_bvh_build_tree_device)
    t_mor, d_mor = device_build_ms(leaves_dev, n, lib.trq_bvh_build_tree_morton_device)
    say(f"{name} device tree build: SAH {t_sah:.3f} ms (maxDepth {d_sah}), Morton {t_mor:.3f} ms (maxDepth {d_mor}), "
        f"{t_sah / t_mor:.1f}x")
    d_tri, d_idx = dev(prim.triList), dev(prim.idxList)
    scene = Scene(DevicePrimitive.build(triList=d_tri, idxList=d_idx), 0)
    t_rb = median_ms(lambda: scene.rebuild(d_tri))
    info_sah = dict(scene.info)
    t_rbm = median_ms(lambda: scene.rebuild(d_tri, method="morton"))
    info_mor = dict(scene.info)
    say(f"{name} trq_scene_rebuild (new device vertices): SAH {t_rb:.2f} ms, TRQ_BUILD_MORTON {t_rbm:.2f} ms, {t_rb / t_rbm:.1f}x")
    rays = rays_to_torch(rays_np, "cuda:0")
    hits = torch.empty((rays.shape[0], 8), dtype=torch.float32, device="cuda")
    from tracer_b200.scene import Primitive
    for method, info in (("sah", info_sah), ("morton", info_mor)):
        scene.rebuild(method=method)
        ms = median_ms(lambda: scene.hit(rays, out=hits), reps=10, events=True)
        got = hits.cpu().numpy().view(L.hit_dtype).reshape(-1)
        tree = Primitive(triList=prim.triList, idxList=prim.idxList, bvhList=scene.bvh())
        checked = oracle_check(port, tree, rays_np, got, f"{name} {method}")
        say(f"{name} closest-hit through the {method} tree: {rays.shape[0] / ms / 1e3:.0f} Mrays/s ({ms:.3f} ms), maxDepth "
            f"{info['maxDepth']}, {info['nNode']} nodes; {checked} sampled hits equal the oracle")
    scene.close()
    return t_rb, t_rbm


def profile_morton_rebuild(prim):
    d_tri, d_idx = dev(prim.triList), dev(prim.idxList)
    scene = Scene(DevicePrimitive.build(triList=d_tri, idxList=d_idx), 0)
    scene.rebuild(d_tri, method="morton")
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    reps = 5
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        for _ in range(reps):
            scene.rebuild(d_tri, method="morton")
        torch.cuda.synchronize()
    per = {}
    for e in p.events():
        if e.device_type.name == "CUDA":
            k = e.name if len(e.name) < 70 else e.name[:67] + "..."
            per.setdefault(k, [0.0, 0])
            per[k][0] += e.device_time / 1e3 if hasattr(e, "device_time") else e.cuda_time / 1e3
            per[k][1] += 1
    say(f"C3 Morton rebuild, device time per kernel and copy (torch.profiler, mean of {reps} rebuilds):")
    total = 0.0
    for k, (ms, cnt) in sorted(per.items(), key=lambda kv: -kv[1][0]):
        total += ms / reps
        say(f"  {ms / reps:8.4f} ms  x{cnt / reps:4.0f}  {k}")
    say(f"  {total:8.4f} ms  total device time per rebuild")
    scene.close()


def main():
    assert torch.cuda.is_available(), "morton_perf.py measures on a GPU"
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    say(f"device 0: {gpu}")
    from oracle.pyoracle import Port
    port = Port()

    c3 = H.scene_c3(2)
    s = Scene(c3, 0)
    primary = H.cornell_camera_rays(3840, 2160)
    d_primary = rays_to_torch(primary, "cuda:0")
    recs = s.expand(d_primary, s.hit(d_primary)).cpu().numpy().view(L.record_dtype).reshape(-1)
    s.close()
    bounce = H.bounce_rays(recs, 0)[0]
    rb = compare("C3", c3, bounce, port)

    soup = H.scene_soup(1_000_000, seed=1, extent=0.004)
    compare("soup 1M", soup, H.random_rays(1 << 22, seed=7), port)
    profile_morton_rebuild(c3)
    say(f"C3 rebuild speed-up with TRQ_BUILD_MORTON: {rb[0] / rb[1]:.1f}x")


if __name__ == "__main__":
    main()
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write("# python tools/morton_perf.py (one run; medians of the repetitions)\n" + "\n".join(lines) + "\n")
