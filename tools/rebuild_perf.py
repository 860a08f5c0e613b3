#!/usr/bin/env python
"""Developer tool: device leaves, rebuild and refit times, and what a rebuild buys the traversal after large motion.
Usage: python tools/rebuild_perf.py [out.txt]      (prints the report; also writes it to out.txt when given)

  1. BVH::buildNode for the 1.0 M triangles of C3: trq_bvh_build_nodes_triangles_device (CUDA events) against the host's
     trq_bvh_build_nodes_triangles (host clock).
  2. trq_scene_rebuild against trq_scene_update_vertices on C3 (host clock around the synchronous calls).
  3. Closest-hit Mrays/s on 4 M random rays (CUDA events) through a 1 M-triangle soup: as built; after every triangle
     has taken another's place, refit only; after a rebuild.
Every timed call is warmed up first (the refit-only trace, seconds long, runs once after the kernels are warm); every time
is the median of the repetitions."""
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

REPS = 10
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()


def median_ms(fn, reps=REPS, events=False, warm=True):
    if warm:
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        if events:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); b.synchronize()
            out.append(a.elapsed_time(b))
        else:
            torch.cuda.synchronize(); t = time.perf_counter(); fn(); torch.cuda.synchronize()
            out.append(1e3 * (time.perf_counter() - t))
    return float(np.median(out))


assert torch.cuda.is_available(), "rebuild_perf.py measures on a GPU"
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
say(f"device 0: {gpu}")

# 1. leaves
tri, idx = H.cornell_triangle_soup(with_teapot=True, mesh_levels=2, with_coatball=True)
n = idx.size // 3
d_tri, d_idx = dev(tri), dev(idx)
d_out = torch.empty(n * 64, dtype=torch.uint8, device="cuda")
h_out = np.zeros(n, dtype=L.bvh_dtype)
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
t_dev = median_ms(lambda: check(lib.trq_bvh_build_nodes_triangles_device(d_tri.data_ptr(), d_idx.data_ptr(), n, 0, d_out.data_ptr(), 0, st), "leaves"),
                  reps=50, events=True)
t_host = median_ms(lambda: check(lib.trq_bvh_build_nodes_triangles(tri.ctypes.data, idx.ctypes.data, n, 0, h_out.ctypes.data), "leaves"), reps=5)
assert d_out.cpu().numpy().tobytes() == h_out.tobytes()
say(f"C3 leaves ({n} triangles): device {t_dev:.3f} ms, host {t_host:.1f} ms (identical bytes)")

# 2. rebuild vs refit on C3, built on the device
prim = DevicePrimitive.build(triList=d_tri, idxList=d_idx)
scene = Scene(prim, 0)
t_build = median_ms(lambda: DevicePrimitive.build(triList=d_tri, idxList=d_idx), reps=5)
t_rebuild = median_ms(lambda: scene.rebuild(), reps=REPS)
t_rebuild_v = median_ms(lambda: scene.rebuild(d_tri), reps=REPS)
t_refit = median_ms(lambda: scene.update_vertices(d_tri), reps=REPS)
say(f"C3 ({scene.info['nNode']} nodes): DevicePrimitive.build (leaves + tree) {t_build:.2f} ms | rebuild {t_rebuild:.2f} ms, "
    f"rebuild with new device vertices {t_rebuild_v:.2f} ms | update_vertices (refit) {t_refit:.2f} ms")
scene.close()
del prim

# 3. traversal after a large motion: refit against rebuild
soup = H.scene_soup(1_000_000, seed=1, extent=0.004)
rays = rays_to_torch(H.random_rays(1 << 22, seed=7), "cuda:0")
hits = torch.empty((rays.shape[0], 8), dtype=torch.float32, device="cuda")
perm = np.random.default_rng(3).permutation(soup.nTri)
moved = np.ascontiguousarray(soup.triList.reshape(-1, 3)[perm].reshape(-1))
s = Scene(soup, 0)


def rate(label, reps=REPS, warm=True):
    ms = median_ms(lambda: s.hit(rays, out=hits), reps=reps, events=True, warm=warm)
    say(f"soup 1M closest-hit, {label}: {rays.shape[0] / ms / 1e3:.3g} Mrays/s ({ms:.2f} ms for {rays.shape[0]} rays)")


rate("as built")
s.update_vertices(moved)
rate("triangles permuted, refit only", reps=1, warm=False)          # seconds per batch: one run (the kernels are warm)
t_rb = median_ms(lambda: s.rebuild(), reps=3)
rate("triangles permuted, rebuilt")
say(f"soup 1M rebuild {t_rb:.2f} ms")
s.close()

if len(sys.argv) > 1:
    with open(sys.argv[1], "w") as f:
        f.write("# python tools/rebuild_perf.py (one run; medians of the repetitions)\n" + "\n".join(lines) + "\n")
