#!/usr/bin/env python
"""Developer tool for compute-sanitizer runs: one small pass over every kernel family (trace packed in every launch
configuration and both record formats / reflayout, any-hit, sort, resolve, expand, producers, indirect trace, single-rank
gather with both senders' code path, GPU builder host + device resident, device-side scene creation, refit) on the
mixed-primitive Cornell scene."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from tracer_b200 import Scene, harness as H  # noqa: E402
from tracer_b200.scene import BVHBuilder  # noqa: E402

prim = H.scene_reference_cornell()
scene = Scene(prim, 0)
r0 = scene.cast_rays((278, 278, -800), (278, 278, 278), (0, 1, 0), np.float32(45 * (np.pi / 180)), 96, 54)
for refl in (False, True):
    h0 = scene.hit(r0, reflayout=refl)
for c in range(len(Scene.kernel_configs())):                 # every launch configuration, both record formats
    try:
        scene.set_kernel_config(c)
    except Exception:
        continue
    for h16 in (False, True):
        scene.hit(r0, hit16=h16); scene.hit(r0, any=True, hit16=h16)
scene.set_kernel_config(-1)
h0 = scene.hit(r0, sort=True) if r0.shape[0] >= 65536 else scene.hit(r0)
big = torch.cat([r0] * 16)
scene.hit(big, sort=True)
# automatic ordering (probe + the passes that may return at once): needs >= 2^20 rays; an incoherent and a coherent batch
os.environ["TRQ_AUTO_SORT"] = "1"
huge = torch.cat([r0] * 203)
scene.hit(huge)                                                    # camera rays repeated: coherent
scene.hit(huge[torch.randperm(huge.shape[0], device=huge.device)].contiguous())   # shuffled: incoherent
del os.environ["TRQ_AUTO_SORT"]
scene.expand(r0, h0)
r1, s1, c1 = scene.spawn_bounce(r0, h0, seed_base=3)
h1 = scene.hit_indirect(r1, c1)
sh, s2, c2 = scene.spawn_shadow(r1, h1, 5, 6, seed_base=5, count_in=c1)
scene.hit_indirect(sh, c2, any=True)
# the RNG-texture producers (row f-4) and the single-rank gather path (tile counts in the trace, sender kernel, gather_wait_kernel)
tex = torch.randint(-2**31, 2**31 - 1, (r0.shape[0], 4), dtype=torch.int32, device=r0.device)
r2, s3, c3 = scene.spawn_bounce(r0, h0, rng_state=tex)
scene.spawn_shadow(r2, scene.hit_indirect(r2, c3), 5, 6, count_in=c3, pixel_of=s3, rng_state=tex)
from tracer_b200 import dist as D  # noqa: E402
hg = D.HitGather(scene, r0.shape[0])
for k in range(4):
    hg.trace(r0, hit16=False); hits_all, counts = hg.wait()
torch.cuda.synchronize(); hg.status()
assert int(counts[0].item()) == r0.shape[0] and torch.equal(hits_all[0].view(torch.int32), h0.view(torch.int32))
hg.close()
host = scene.hit(H.random_rays(5000, seed=1, lo=(-245, 0, 0), hi=(800, 555, 555)))
b = BVHBuilder(); b.buildNodesTriangles(prim.triList, prim.idxList)
g = b.buildTree(gpu=0)
# device-resident build -> device-resident scene creation -> refit
from tracer_b200 import DevicePrimitive  # noqa: E402
nodes = b.buildTreeDevice(0)
tri = torch.from_numpy(prim.triList.view(np.uint8).reshape(-1).copy()).cuda()
idx = torch.from_numpy(prim.idxList.view(np.uint8).reshape(-1).copy()).cuda()
ds = Scene(DevicePrimitive(triList=tri, idxList=idx, bvhList=nodes), 0)
ds.hit(r0)
ds.update_vertices(tri); ds.hit(r0, any=True)
# the kernels specialised by leaf types: triangles only (ds) and triangles + spheres (C1's spheres), every configuration
sp = Scene(H.scene_c1(), 0)
sp.update_primitives(spheres=torch.from_numpy(H.scene_c1().sphereList.view(np.uint8).reshape(-1).copy()).cuda())   # sphere leaf refit
rs = scene.cast_rays((13, 2, 3), (0, 0, 0), (0, 1, 0), np.float32(20 * np.pi / 180), 96, 54)
for sc, rr in ((ds, r0), (sp, rs)):
    for c in range(len(Scene.kernel_configs())):
        try:
            sc.set_kernel_config(c)
        except Exception:
            continue
        for h16 in (False, True):
            sc.hit(rr, hit16=h16); sc.hit(rr, any=True, hit16=h16)
    sc.set_kernel_config(-1)
dm = Scene(DevicePrimitive.from_host(prim, "cuda:0"), 0)     # mixed leaves through the device planner
assert torch.equal(dm.hit(r0).view(torch.int32), h0.view(torch.int32))
torch.cuda.synchronize()
print("sanitize pass done:", int(c1.item()), int(c2.item()), int((host["flags"] & 1).sum()), g.size)
