#!/usr/bin/env python
"""Developer tool: what moving spheres, squares and cubes of a live scene costs (trq_scene_update_primitives).
Usage: python tools/update_perf.py [out.txt]      (prints the report; also writes it to out.txt when given)

  1. update_primitives moving all 10,012 spheres of C4 (device tensor), against trq_scene_create_device of the same scene
     and against update_vertices on C3 (host clock around the synchronous calls).
  2. C1 animated: every sphere moved, then one 1280 x 720 (921,600-ray) primary trace per frame (host clock per frame).
  3. Closest-hit Mrays/s (CUDA events) on C4 primary rays after an update, against a scene created afresh from the same
     lists and node array: the tree and the packed bytes are the same, so the rates should be too.
Every timed call is warmed up first; every time is the median of the repetitions."""
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from tracer_b200 import DevicePrimitive, Scene, harness as H  # noqa: E402
from tracer_b200.scene import Primitive  # noqa: E402

REPS = 20
lines = []
f32 = np.float32


def say(s):
    print(s, flush=True)
    lines.append(s)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()


def median_ms(fn, reps=REPS, events=False):
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


def moved_spheres(s, rng, d):
    s = s.copy()
    off = rng.uniform(-d, d, (s.size, 3)).astype(f32)
    s["center"] += off
    s["box_mini"] += off
    s["box_maxi"] += off
    return s


assert torch.cuda.is_available(), "update_perf.py measures on a GPU"
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
say(f"device 0: {gpu}")
rng = np.random.default_rng(1)
cam = dict(look_from=(278, 278, -800), look_at=(278, 278, 278), view_up=(0, 1, 0), vfov=f32(45 * np.pi / 180), W=1280, H=720)

# 1. C4: update the spheres against creating the scene again; C3 refit for scale
c4 = H.scene_c4()
scene = Scene(c4, 0)
frames = [dev(moved_spheres(c4.sphereList, rng, 3)) for _ in range(2)]
k = [0]


def update_c4():
    k[0] ^= 1
    scene.update_primitives(spheres=frames[k[0]])


t_update = median_ms(update_c4)
dprim = DevicePrimitive.from_host(c4, "cuda:0")
t_create = median_ms(lambda: Scene(dprim, 0).close(), reps=5)
say(f"C4 ({scene.info['nNode']} nodes, {c4.sphereList.size} spheres, {c4.nTri} triangles): update_primitives(all spheres, device) "
    f"{t_update:.2f} ms | trq_scene_create_device of the same scene {t_create:.2f} ms")
c3 = Scene(H.scene_c3(), 0)
d_verts = dev(c3.primitives.triList)
t_refit = median_ms(lambda: c3.update_vertices(d_verts))
say(f"C3 ({c3.info['nNode']} nodes): update_vertices (refit) {t_refit:.2f} ms")
c3.close()

# 3. (on the C4 scene as updated) trace rate after an update against a fresh scene of the same lists and tree
scene.update_primitives(spheres=frames[0])
rays = scene.cast_rays(**cam)
hits = torch.empty((rays.shape[0], 8), dtype=torch.float32, device="cuda")
r_upd = median_ms(lambda: scene.hit(rays, out=hits), events=True)
fresh = Scene(Primitive(sphereList=frames[0].cpu().numpy().view(c4.sphereList.dtype), squareList=c4.squareList, triList=c4.triList,
                        idxList=c4.idxList, bvhList=scene.bvh()), 0)
hits2 = torch.empty_like(hits)
r_fresh = median_ms(lambda: fresh.hit(rays, out=hits2), events=True)
assert torch.equal(hits.view(torch.int32), hits2.view(torch.int32))
say(f"C4 closest-hit, {rays.shape[0]} primary rays: after update {rays.shape[0] / r_upd / 1e3:.4g} Mrays/s ({r_upd:.3f} ms) | "
    f"fresh scene {rays.shape[0] / r_fresh / 1e3:.4g} Mrays/s ({r_fresh:.3f} ms) (identical hits)")
fresh.close()
scene.close()
del dprim

# 2. C1 animated: move every sphere, then trace one primary frame
c1 = H.scene_c1()
s1 = Scene(c1, 0)
c1_frames = [dev(moved_spheres(c1.sphereList, rng, 0.2)) for _ in range(2)]
c1_cam = dict(look_from=(13, 2, 3), look_at=(0, 0, 0), view_up=(0, 1, 0), vfov=f32(20 * np.pi / 180), W=1280, H=720)
rays1 = s1.cast_rays(**c1_cam)
hits1 = torch.empty((rays1.shape[0], 8), dtype=torch.float32, device="cuda")
j = [0]


def c1_update():
    j[0] ^= 1
    s1.update_primitives(spheres=c1_frames[j[0]])


def c1_frame():
    c1_update()
    s1.hit(rays1, out=hits1)


t1_update = median_ms(c1_update)
t1_trace = median_ms(lambda: s1.hit(rays1, out=hits1))
t1_frame = median_ms(c1_frame)
say(f"C1 ({s1.info['nNode']} nodes, {c1.sphereList.size} spheres): update_primitives(all spheres) {t1_update:.3f} ms | "
    f"{rays1.shape[0]}-ray primary trace {t1_trace:.3f} ms | frame (update + trace) {t1_frame:.3f} ms")
s1.close()

if len(sys.argv) > 1:
    with open(sys.argv[1], "w") as f:
        f.write("# python tools/update_perf.py (one run; medians of the repetitions)\n" + "\n".join(lines) + "\n")
