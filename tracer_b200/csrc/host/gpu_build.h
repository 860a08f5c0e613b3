// tracer_b200/csrc/host/gpu_build.h -- the GPU builder's pieces that scene rebuilds (trq_api.cu) call directly.
// Implemented in bvh_build_gpu.cu; everything runs on the legacy default stream of the current device.
#pragma once
#include <stdint.h>

#include "layout.h"
#include "scratch.h"

namespace trq {

// dLeaves[0..n) -> dOut[0..2n-1): root at 0, leaves at 1..n in list order, interiors after (BVH.hh:263-268). n >= 2.
// Interior depth above 31 still builds the whole tree and returns TRQ_ERR_DEPTH with its true depth.
int build_on_device(const RefBVH* dLeaves, uint32_t n, RefBVH* dOut, int device, uint32_t* maxDepthOut);

// The same output layout from the Morton builder (kernels/morton_build.cuh). n >= 2. Interior depth is at most 31.
int build_morton_on_device(const RefBVH* dLeaves, uint32_t n, RefBVH* dOut, int device, uint32_t* maxDepthOut);

// The leaf list of a rebuild: the nLeaf leaves the root reaches (ref[i] != TRQ_REF_DONE_WORD) in bvhList order, into
// *leavesOut (allocated from `mem`). Triangle leaves are made again from `verts`; the others keep pType, pIndex and box.
int reachable_leaves_on_device(const RefBVH* bvh, const uint32_t* ref, uint32_t nNode, uint32_t nLeaf, const RefVertex* verts,
                               const uint32_t* idx, PoolScratch& mem, RefBVH** leavesOut);

// The leaf refit of trq_scene_update_primitives: every leaf the root reaches whose kind has a non-NULL list (the scene's
// replaced records) gets the box trq_bvh_build_node gives for its record; only mini / maxi are written.
int refit_primitive_leaves_on_device(RefBVH* bvh, const uint32_t* ref, uint32_t nNode, const RefSphere* spheres, const RefSquare* squares,
                                     const RefCube* cubes);

}  // namespace trq
