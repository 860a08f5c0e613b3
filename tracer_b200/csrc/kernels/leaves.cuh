// tracer_b200/csrc/kernels/leaves.cuh -- BVH::buildNode (BVH.hh:271-314) on the GPU: the leaf records of
// trq_bvh_build_nodes_triangles / trq_bvh_build_node, bit for bit, the leaf list of a scene rebuild, and the leaf refit
// of trq_scene_update_primitives.
//
// The host restatement (csrc/host/bvh_build.cpp) is compiled without contraction and calls glibc's fminf / fmaxf, which
// return the OTHER argument when one is NaN and the FIRST argument when the two compare equal (-0.0 vs +0.0). The
// triangle box is std::min / std::max over {a, b, c}: the first of the smallest (largest) under `<`, so a NaN in front
// wins and a NaN behind is skipped. The functions below spell those rules out rather than rely on CUDA's fminf / fmaxf,
// which make no promise about which zero they return.
#pragma once
#include <cfloat>
#include <cstddef>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../../include/tracer_rq.h"
#include "../host/layout.h"
#include "scene_dev.cuh"
#include "strict_math.cuh"

namespace trq {
namespace leaves {

__device__ __forceinline__ float host_fminf(float a, float b) { return (b < a || a != a) ? b : a; }
__device__ __forceinline__ float host_fmaxf(float a, float b) { return (a < b || a != a) ? b : a; }

// BVH::buildNode: world AABB of the 8 corners of [lo, hi] under the column-major model matrix m (never NULL: the
// identity is multiplied out like any other matrix, so 0 * inf gives NaN as on the host).
__device__ __forceinline__ void build_node(const float lo[3], const float hi[3], const float m[16], int32_t pType, uint32_t pIndex,
                                           RefBVH* out) {
    float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    const float* ele[2] = {lo, hi};
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const float x = ele[i][0], y = ele[j][1], z = ele[k][2];
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float t = fadd(fadd(fadd(fmul(m[0 + c], x), fmul(m[4 + c], y)), fmul(m[8 + c], z)), fmul(m[12 + c], 1.0f));
                    mn[c] = host_fminf(mn[c], t);
                    mx[c] = host_fmaxf(mx[c], t);
                }
            }
    RefBVH nb = {};
    nb.pType = pType;
    nb.pIndex = pIndex;
    for (int c = 0; c < 3; ++c) { nb.bBOX.mini[c] = mn[c]; nb.bBOX.maxi[c] = mx[c]; }
    *out = nb;
}

// Leaf of triangle p (AAPLRenderer.mm:575-589): std::min / std::max of its three vertices, identity model.
__device__ __forceinline__ void triangle_leaf(const RefVertex* __restrict__ verts, const uint32_t* __restrict__ idx, uint32_t p,
                                              uint32_t pIndex, RefBVH* out) {
    const float* a = verts[idx[3 * (size_t)p]].v;
    const float* b = verts[idx[3 * (size_t)p + 1]].v;
    const float* c = verts[idx[3 * (size_t)p + 2]].v;
    float lo[3], hi[3];
    for (int k = 0; k < 3; ++k) {
        float l = a[k], h = a[k];
        if (b[k] < l) l = b[k];
        if (c[k] < l) l = c[k];
        if (h < b[k]) h = b[k];
        if (h < c[k]) h = c[k];
        lo[k] = l; hi[k] = h;
    }
    const float ident[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    build_node(lo, hi, ident, TRQ_TRIANGLE, pIndex, out);
}

__global__ void __launch_bounds__(256)
triangle_leaves_kernel(const RefVertex* __restrict__ verts, const uint32_t* __restrict__ idx, uint32_t nTri, uint32_t pIndexBase, RefBVH* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nTri) triangle_leaf(verts, idx, i, pIndexBase + i, &out[i]);
}

// Where BVH::buildNode's arguments sit in a Sphere / Square / Cube record (AAPLRenderer.mm:454-468): `stride` bytes each,
// the model matrix at byte modelAt and the AABB at byte boxAt (boundingBOX, or box for a Cube). False for any other pType.
inline bool record_layout(int32_t pType, uint32_t* stride, uint32_t* modelAt, uint32_t* boxAt) {
    switch (pType) {
        case TRQ_SPHERE: *stride = sizeof(RefSphere); *modelAt = offsetof(RefSphere, model); *boxAt = offsetof(RefSphere, boundingBOX); return true;
        case TRQ_SQUARE: *stride = sizeof(RefSquare); *modelAt = offsetof(RefSquare, model); *boxAt = offsetof(RefSquare, boundingBOX); return true;
        case TRQ_CUBE:   *stride = sizeof(RefCube);   *modelAt = offsetof(RefCube, model);   *boxAt = offsetof(RefCube, box); return true;
        default: return false;
    }
}

__device__ __forceinline__ void primitive_leaf(const uint8_t* rec, uint32_t modelAt, uint32_t boxAt, int32_t pType, uint32_t pIndex, RefBVH* out) {
    const RefAABB box = *reinterpret_cast<const RefAABB*>(rec + boxAt);
    float m[16];
    for (int k = 0; k < 16; ++k) m[k] = reinterpret_cast<const float*>(rec + modelAt)[k];
    build_node(box.mini, box.maxi, m, pType, pIndex, out);
}

__global__ void __launch_bounds__(256)
primitive_leaves_kernel(const uint8_t* __restrict__ list, uint32_t n, uint32_t stride, uint32_t modelAt, uint32_t boxAt, int32_t pType,
                        uint32_t pIndexBase, RefBVH* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) primitive_leaf(list + (size_t)i * stride, modelAt, boxAt, pType, pIndexBase + i, &out[i]);
}

// ---- leaf refit of trq_scene_update_primitives: the record list of each kind, indexed by pType (TRQ_SPHERE, TRQ_SQUARE,
// TRQ_CUBE); list == nullptr keeps the leaves of that kind.
struct RecordList { const uint8_t* list; uint32_t stride, modelAt, boxAt; };
struct RecordLists { RecordList kind[3]; };

// Every leaf the root reaches (ref[i] != TRQ_REF_DONE_WORD) whose kind was replaced gets the box trq_bvh_build_node gives
// for its record list[pIndex]. Only mini / maxi are written: links, pType, pIndex and the padding words stay as they are.
__global__ void __launch_bounds__(256)
refit_primitive_leaves_kernel(RefBVH* N, const uint32_t* __restrict__ ref, uint32_t n, RecordLists lists) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || ref[i] == TRQ_REF_DONE_WORD) return;
    const int32_t t = N[i].pType;
    if (t != TRQ_SPHERE && t != TRQ_SQUARE && t != TRQ_CUBE) return;
    // (constant indices: a dynamic index would copy the parameter block to local memory)
    const RecordList r = t == TRQ_SPHERE ? lists.kind[TRQ_SPHERE] : t == TRQ_SQUARE ? lists.kind[TRQ_SQUARE] : lists.kind[TRQ_CUBE];
    if (!r.list) return;
    const uint32_t p = N[i].pIndex;
    RefBVH nb;
    primitive_leaf(r.list + (size_t)p * r.stride, r.modelAt, r.boxAt, t, p, &nb);
    for (int k = 0; k < 3; ++k) { N[i].bBOX.mini[k] = nb.bBOX.mini[k]; N[i].bBOX.maxi[k] = nb.bBOX.maxi[k]; }
}

// ---- leaf list of trq_scene_rebuild: every leaf the root reaches (ref != TRQ_REF_DONE_WORD), in bvhList order
__global__ void __launch_bounds__(256)
reachable_leaf_flag_kernel(const RefBVH* __restrict__ N, const uint32_t* __restrict__ ref, uint32_t n, uint32_t* flag) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    flag[i] = (i < n && ref[i] != TRQ_REF_DONE_WORD && N[i].pType != TRQ_BVH) ? 1u : 0u;   // flag[n] = 0
}

// Leaf pos[i] of the list: a triangle is made again from the current vertices keeping its pIndex; any other leaf keeps
// pType, pIndex and box. Every other field is zero, as trq_bvh_build_node writes it.
__global__ void __launch_bounds__(256)
reachable_leaf_scatter_kernel(const RefBVH* __restrict__ N, const uint32_t* __restrict__ flag, const uint32_t* __restrict__ pos, uint32_t n,
                              const RefVertex* __restrict__ verts, const uint32_t* __restrict__ idx, RefBVH* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !flag[i]) return;
    const RefBVH b = N[i];
    if (b.pType == TRQ_TRIANGLE) { triangle_leaf(verts, idx, b.pIndex, b.pIndex, &out[pos[i]]); return; }
    RefBVH nb = {};
    nb.pType = b.pType;
    nb.pIndex = b.pIndex;
    for (int c = 0; c < 3; ++c) { nb.bBOX.mini[c] = b.bBOX.mini[c]; nb.bBOX.maxi[c] = b.bBOX.maxi[c]; }
    out[pos[i]] = nb;
}

}  // namespace leaves
}  // namespace trq
