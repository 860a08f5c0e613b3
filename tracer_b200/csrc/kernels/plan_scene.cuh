// tracer_b200/csrc/kernels/plan_scene.cuh -- validation and numbering of a reference-layout BVH ON THE DEVICE.
//
// trq_scene_create walks the tree once on the host (plan_layout in trq_api.cu) to validate the layout contract of
// BVH.hh:15-22 / Render.hh:135-252 and to assign every node its packed reference. When the node array already lives on
// the GPU (trq_scene_create_device: the output of trq_bvh_build_tree_device, or a caller's own device builder) the same
// plan is computed here without a device-to-host copy of the tree, and must give the SAME references:
//   leaves     numbered per kind in depth-first order, left child first;
//   interior   the first packed::kTopMax of a breadth-first walk come first in that order (the block a kernel may stage in shared
//              memory), the others follow in depth-first (pre-)order.
// Depth-first positions need no traversal: with cnt[x] = (interior nodes, triangle / sphere / square leaves) below x,
//   pre(x)   = depth(x) + sum over ancestors a with x in right(a) of cnt[left(a)].interior
//   slot_k(x) =           sum over ancestors a with x in right(a) of cnt[left(a)].k
// so one bottom-up pass (arrival counters, Karras-style) and one climb per node do it.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../../include/tracer_rq.h"
#include "../host/layout.h"
#include "packed_layout.cuh"
#include "scene_dev.cuh"

namespace trq {
namespace plan {

enum : uint32_t { ERR_NONE = 0, ERR_CHILD_RANGE, ERR_CHILDREN, ERR_PARENT_LINK, ERR_ROOT_PARENT, ERR_LEAF_INDEX, ERR_VERTEX_INDEX,
                  ERR_DEPTH, ERR_UNREACHABLE };

struct PlanInfo {
    uint32_t error, errorNode, errorA, errorB;     // first error wins (atomicCAS on `error`)
    uint32_t maxDepth, maxPIndex, nTop, rootRef;
    uint32_t nInterior, nLeaf, nTri, nSphere, nSquare, pad[3];
    float    rootMin[4], rootMax[4];
};

struct Counts { uint32_t interior, tri, sph, sq; };     // 16 B, one per node

__device__ __forceinline__ void raise(PlanInfo* info, uint32_t code, uint32_t node, uint32_t a = 0, uint32_t b = 0) {
    if (atomicCAS(&info->error, 0u, code) == 0u) { info->errorNode = node; info->errorA = a; info->errorB = b; }
}

// One thread per node: the local checks of plan_layout (child indices, parent back-links, primitive indices).
__global__ void __launch_bounds__(256)
validate_kernel(const RefBVH* __restrict__ N, uint32_t n, uint32_t nSphere, uint32_t nSquare, uint32_t nCube, uint32_t nTri, uint32_t nVert,
                const uint32_t* __restrict__ idx, PlanInfo* info) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const RefBVH b = N[i];
    if (i == 0) {
        if (b.parent != 0) raise(info, ERR_ROOT_PARENT, 0, b.parent);
        for (int k = 0; k < 3; ++k) { info->rootMin[k] = b.bBOX.mini[k]; info->rootMax[k] = b.bBOX.maxi[k]; }
    } else {
        // every other node must hang under the parent it names (no orphans, no second parents)
        const uint32_t p = b.parent;
        if (p >= n || N[p].pType != TRQ_BVH || (N[p].left != i && N[p].right != i)) raise(info, ERR_PARENT_LINK, i, p);
    }
    if (b.pType == TRQ_BVH) {
        if (b.left >= n || b.right >= n) { raise(info, ERR_CHILD_RANGE, i, b.left, b.right); return; }
        if (b.left == 0 || b.right == 0 || b.left == b.right) { raise(info, ERR_CHILDREN, i, b.left, b.right); return; }
        if (N[b.left].parent != i || N[b.right].parent != i) raise(info, ERR_PARENT_LINK, i, N[b.left].parent, N[b.right].parent);
    } else {
        atomicMax(&info->maxPIndex, b.pIndex);
        if (b.pType == TRQ_TRIANGLE) {
            if (b.pIndex >= nTri) { raise(info, ERR_LEAF_INDEX, i, b.pIndex, nTri); return; }
            for (int k = 0; k < 3; ++k)
                if (idx[3 * (size_t)b.pIndex + k] >= nVert) raise(info, ERR_VERTEX_INDEX, i, b.pIndex);
        } else if (b.pType == TRQ_SPHERE) { if (b.pIndex >= nSphere) raise(info, ERR_LEAF_INDEX, i, b.pIndex, nSphere); }
        else if (b.pType == TRQ_SQUARE)   { if (b.pIndex >= nSquare) raise(info, ERR_LEAF_INDEX, i, b.pIndex, nSquare); }
        else if (b.pType == TRQ_CUBE)     { if (b.pIndex >= nCube) raise(info, ERR_LEAF_INDEX, i, b.pIndex, nCube); }
    }
}

// Bottom-up subtree counts. One thread per node; leaves start a climb, the second arrival at an interior node merges its
// two children. `prev != 1` also ends a climb that would go round a cycle of mutually consistent links.
__global__ void __launch_bounds__(256)
counts_kernel(const RefBVH* __restrict__ N, uint32_t n, Counts* cnt, uint32_t* leafTotal, uint32_t* arrivals) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || N[i].pType == TRQ_BVH) return;
    Counts c = {0u, N[i].pType == TRQ_TRIANGLE ? 1u : 0u, N[i].pType == TRQ_SPHERE ? 1u : 0u, N[i].pType == TRQ_SQUARE ? 1u : 0u};
    cnt[i] = c; leafTotal[i] = 1u;
    if (i == 0) return;                                            // single-leaf scene
    uint32_t node = N[i].parent;
    for (int guard = 0; guard < 64; ++guard) {
        if (node >= n) return;                                      // broken links: reported by validate_kernel, never dereferenced
        __threadfence();
        if (atomicAdd(&arrivals[node], 1u) != 1u) return;           // first child to arrive waits for its sibling
        const uint32_t l = N[node].left, r = N[node].right;
        if (l >= n || r >= n) return;
        // __ldcg: the children's counts were written by other SMs in this launch
        const uint4 a = __ldcg(reinterpret_cast<const uint4*>(&cnt[l])), b = __ldcg(reinterpret_cast<const uint4*>(&cnt[r]));
        Counts m = {a.x + b.x + 1u, a.y + b.y, a.z + b.z, a.w + b.w};
        cnt[node] = m;
        leafTotal[node] = __ldcg(&leafTotal[l]) + __ldcg(&leafTotal[r]);
        if (node == 0) return;
        node = N[node].parent;
    }
}

// One thread per node: climb to the root accumulating depth and depth-first offsets; leaves get their final reference,
// interior nodes their pre-order position (turned into a reference by refs_kernel once the breadth-first block is known).
__global__ void __launch_bounds__(256)
number_kernel(const RefBVH* __restrict__ N, uint32_t n, const Counts* __restrict__ cnt, const uint32_t* __restrict__ leafTotal,
              uint32_t* ref, uint32_t* pre, PlanInfo* info) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (i == 0) {
        const Counts c = cnt[0];
        info->nInterior = c.interior; info->nLeaf = leafTotal[0]; info->nTri = c.tri; info->nSphere = c.sph; info->nSquare = c.sq;
        if (c.interior + leafTotal[0] != n) raise(info, ERR_UNREACHABLE, 0, c.interior + leafTotal[0], n);   // orphaned / cyclic components
    }
    uint32_t depth = 0;
    Counts off = {0u, 0u, 0u, 0u};
    uint32_t x = i;
    while (x != 0) {
        if (depth > 40) { raise(info, ERR_DEPTH, i, depth); return; }
        const uint32_t a = N[x].parent;
        if (a >= n) return;                                        // reported by validate_kernel
        if (N[a].right == x && N[a].left < n) {
            const Counts c = cnt[N[a].left];
            off.interior += c.interior; off.tri += c.tri; off.sph += c.sph; off.sq += c.sq;
        }
        x = a; ++depth;
    }
    const int32_t t = N[i].pType;
    if (t == TRQ_BVH) {
        if (depth > 31) { raise(info, ERR_DEPTH, i, depth); return; }   // the reference's trail has 32 bits (Render.hh:140)
        atomicMax(&info->maxDepth, depth);
        pre[i] = depth + off.interior;
    } else {
        pre[i] = 0xffffffffu;
        ref[i] = t == TRQ_TRIANGLE ? TRQ_MAKE_REF(REF_TRI, off.tri)
               : t == TRQ_SPHERE   ? TRQ_MAKE_REF(REF_SPHERE, off.sph)
               : t == TRQ_SQUARE   ? TRQ_MAKE_REF(REF_SQUARE, off.sq)
               : t == TRQ_CUBE     ? TRQ_MAKE_REF(REF_CUBE, i) : TRQ_MAKE_REF(REF_NOP, i);
    }
}

// One CTA: breadth-first walk of the interior nodes from the root, level by level, left to right, until packed::kTopMax nodes
// are listed (the queue order of plan_layout's walk). topPos[node] = position + 1; sortedPre = their pre-order positions,
// ascending (refs_kernel counts how many of them precede a node).
__global__ void __launch_bounds__(1024)
top_block_kernel(const RefBVH* __restrict__ N, uint32_t n, const uint32_t* __restrict__ pre, uint32_t* topPos, uint32_t* sortedPre, PlanInfo* info) {
    auto interior = [&](uint32_t x) { return x < n && N[x].pType == TRQ_BVH; };   // x >= n: broken link, reported by validate_kernel
    __shared__ uint32_t frontier[2][2048];
    __shared__ uint32_t scan[2048];
    __shared__ uint32_t keys[2048];
    __shared__ uint32_t total, nFront, nextFront;
    const uint32_t t = threadIdx.x;
    if (t == 0) { total = 0; nFront = (N[0].pType == TRQ_BVH) ? 1u : 0u; frontier[0][0] = 0u; }
    __syncthreads();
    int cur = 0;
    while (nFront > 0 && total < packed::kTopMax) {
        const uint32_t nf = nFront, base = total;
        // list this level (clipped to the capacity)
        for (uint32_t k = t; k < nf; k += 1024) {
            if (base + k < packed::kTopMax) { topPos[frontier[cur][k]] = base + k + 1; keys[base + k] = pre[frontier[cur][k]]; }
        }
        // children that are interior, in order: exclusive scan of (left interior) + (right interior)
        for (uint32_t k = t; k < 2048; k += 1024) {
            uint32_t c = 0;
            if (k < nf) { const RefBVH& b = N[frontier[cur][k]]; c = (interior(b.left) ? 1u : 0u) + (interior(b.right) ? 1u : 0u); }
            scan[k] = c;
        }
        __syncthreads();
        for (uint32_t off = 1; off < 2048; off <<= 1) {             // Hillis-Steele inclusive scan, two elements per thread
            uint32_t v0 = t >= off ? scan[t - off] : 0u, v1 = (t + 1024) >= off ? scan[t + 1024 - off] : 0u;
            __syncthreads();
            scan[t] += v0; scan[t + 1024] += v1;
            __syncthreads();
        }
        const uint32_t listed = (base + nf < packed::kTopMax) ? nf : (packed::kTopMax - base);
        const uint32_t room = packed::kTopMax - (base + listed);         // what the next level may still add
        for (uint32_t k = t; k < nf; k += 1024) {
            const RefBVH& b = N[frontier[cur][k]];
            uint32_t pos = scan[k] - ((interior(b.left) ? 1u : 0u) + (interior(b.right) ? 1u : 0u));
            if (interior(b.left))  { if (pos < room && pos < 2048u) frontier[cur ^ 1][pos] = b.left; ++pos; }
            if (interior(b.right)) { if (pos < room && pos < 2048u) frontier[cur ^ 1][pos] = b.right; }
        }
        __syncthreads();
        if (t == 0) {
            total = base + listed;
            const uint32_t produced = scan[2047];
            nextFront = produced < room ? produced : room;
            nFront = nextFront;
        }
        __syncthreads();
        cur ^= 1;
    }
    const uint32_t T = total;
    // bitonic sort of the listed nodes' pre-order positions (padded with ~0)
    for (uint32_t k = t; k < 2048; k += 1024) if (k >= T) keys[k] = 0xffffffffu;
    __syncthreads();
    for (uint32_t size = 2; size <= 2048; size <<= 1) {
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            for (uint32_t k = t; k < 1024; k += 1024) {
                const uint32_t lo = 2 * k - (k & (stride - 1));     // index of the lower element of pair k
                const uint32_t hi = lo + stride;
                const bool up = (lo & size) == 0;
                const uint32_t a = keys[lo], b = keys[hi];
                if ((a > b) == up) { keys[lo] = b; keys[hi] = a; }
            }
            __syncthreads();
        }
    }
    for (uint32_t k = t; k < 2048; k += 1024) sortedPre[k] = keys[k];
    if (t == 0) info->nTop = T;
}

// Interior references: breadth-first block first, the rest in pre-order behind it.
__global__ void __launch_bounds__(256)
refs_kernel(const RefBVH* __restrict__ N, uint32_t n, const uint32_t* __restrict__ pre, const uint32_t* __restrict__ topPos,
            const uint32_t* __restrict__ sortedPre, uint32_t* ref, PlanInfo* info) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (N[i].pType == TRQ_BVH) {
        const uint32_t T = info->nTop;
        if (topPos[i]) ref[i] = TRQ_MAKE_REF(REF_INTERIOR, topPos[i] - 1u);
        else {
            const uint32_t p = pre[i];
            uint32_t lo = 0, hi = T;                                // number of listed nodes with a smaller pre-order position
            while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (sortedPre[mid] < p) lo = mid + 1; else hi = mid; }
            ref[i] = TRQ_MAKE_REF(REF_INTERIOR, T + p - lo);
        }
    }
    if (i == 0) info->rootRef = ref[0];
}

// ---- refit (trq_scene_update_vertices): leaf boxes of triangle leaves from the moved vertices (AAPLRenderer.mm:575-589:
// min / max of the three vertices), then interior boxes bottom-up as unions of their children (AABB::make, AABB.hh:227-239;
// BVH.hh:229-231), same arrival-counter climb as above. Only nodes the root reaches take part (ref[i] != TRQ_REF_DONE_WORD):
// trq_scene_create keeps unreachable nodes without checking their fields, and a climb from one of them would give a real
// interior node a third arrival (merged before one child subtree is refit) or leave the arrays.
__global__ void __launch_bounds__(256)
refit_leaves_kernel(RefBVH* N, const uint32_t* __restrict__ ref, uint32_t n, const RefVertex* __restrict__ verts, const uint32_t* __restrict__ idx) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || ref[i] == TRQ_REF_DONE_WORD || N[i].pType != TRQ_TRIANGLE) return;
    const uint32_t p = N[i].pIndex;
    const float* a = verts[idx[3 * (size_t)p]].v; const float* b = verts[idx[3 * (size_t)p + 1]].v; const float* c = verts[idx[3 * (size_t)p + 2]].v;
    for (int k = 0; k < 3; ++k) {
        N[i].bBOX.mini[k] = fminf(fminf(a[k], b[k]), c[k]);
        N[i].bBOX.maxi[k] = fmaxf(fmaxf(a[k], b[k]), c[k]);
    }
}

__global__ void __launch_bounds__(256)
refit_interior_kernel(RefBVH* N, const uint32_t* __restrict__ ref, uint32_t n, uint32_t* arrivals) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || i == 0 || ref[i] == TRQ_REF_DONE_WORD || N[i].pType == TRQ_BVH) return;   // node 0: a one-leaf scene
    uint32_t node = N[i].parent;
    for (int guard = 0; guard < 64; ++guard) {
        __threadfence();
        if (atomicAdd(&arrivals[node], 1u) != 1u) return;
        const RefBVH* l = &N[N[node].left];
        const RefBVH* r = &N[N[node].right];
        for (int k = 0; k < 3; ++k) {                               // __ldcg: child boxes were written by other SMs in this launch
            N[node].bBOX.mini[k] = fminf(__ldcg(&l->bBOX.mini[k]), __ldcg(&r->bBOX.mini[k]));
            N[node].bBOX.maxi[k] = fmaxf(__ldcg(&l->bBOX.maxi[k]), __ldcg(&r->bBOX.maxi[k]));
        }
        if (node == 0) return;
        node = N[node].parent;
    }
}

}  // namespace plan
}  // namespace trq
