// tracer_b200/csrc/kernels/morton_build.cuh -- the Morton-order (LBVH) tree builder on the GPU.
//
// A second builder beside the binned-SAH one (kernels/bvh_build.cuh): one code pass, one sort, at most 32 split launches
// and one refit, with no host round trip per level. It writes the reference's node format (struct BVH, BVH.hh:15-22), so
// planning, packing, traversal, refit and everything downstream take its trees unchanged. The tree it builds is defined
// by the rules below; the sequential host restatement (host/morton_build.cpp) follows the same rules, and the two agree
// byte for byte.
//
//   centroid   centroid_of (AABB::centroid, AABB.hh:22-25) of each leaf's box.
//   quantise   per axis, in strict fp32: lo / hi = min / max of the FINITE centroid components on that axis, ext = hi - lo.
//                q(c) = 2^21 - 1                                      if c is NaN or +inf
//                       0                                             if c is -inf
//                       0                                             if the axis has no finite component, or
//                                                                       ext is not (finite and > 0)
//                       min(2^21 - 1, floor(((c - lo) / ext) * 2^21)) otherwise (c - lo >= 0, so the floor is >= 0)
//              each operation one IEEE round-to-nearest step, in exactly that order (quantise() below).
//   code       63 bits: bit 3i+2 is bit i of qx, bit 3i+1 of qy, bit 3i of qz.
//   order      the leaves sorted by (code, list position): a unique order.
//   topology   top-down. A node at interior depth d (root 0) spanning sorted positions [a, b], m = b - a + 1 >= 2:
//                code[a] == code[b]: the left child gets floor(m / 2) leaves;
//                otherwise the left child gets the positions whose code has the highest bit in which code[a] and code[b]
//                differ clear (Karras 2012), found by binary search.
//              That left size s is then clamped into [m - 2^(31-d), 2^(31-d)], intersected with [1, m - 1]. A node at depth
//              d spans at most 2^(32-d) leaves (the root at most 2^30), so the interval is never empty and each child spans
//              at most 2^(31-d): a node at depth 31 has two leaf children, and the deepest interior level is at most 31 for
//              every input. Where the Morton split already satisfies the clamp, the clamp changes nothing.
//   numbering  the root is node 0; leaves at 1..n in LIST order (BVH.hh:265); the interior node whose split lies between
//              sorted positions g and g + 1 is node n + 1 + g if g < g_root, else n + g (each gap g in [0, n - 2] is split
//              exactly once, g_root by the root). No numbering depends on the order in which threads emit nodes.
//   fields     left / right / parent final indices; axis = the dimension of the highest differing bit of the node's two end
//              codes (0 when they are equal); pType TRQ_BVH, pIndex 0, padding 0; box = union of the two child boxes,
//              bottom-up (gpubuild::refit_kernel). Leaves keep every field but parent.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../../include/tracer_rq.h"
#include "../host/layout.h"
#include "bvh_build.cuh"
#include "strict_math.cuh"

namespace trq {
namespace morton {

constexpr uint32_t kQuantMax = (1u << 21) - 1;
constexpr uint32_t kMaxLevels = 32;             // interior depths 0..31
constexpr uint32_t kLevelCounts = 0;            // counters[0..32]: open nodes of each level (33: none ever opens)
constexpr uint32_t kRootGap = 33;               // counters[33]: the root's split gap
constexpr uint32_t kMaxDepth = 34;              // counters[34]: deepest interior level emitted
constexpr uint32_t kOverflow = 35;              // counters[35]: a level table or the depth bound overflowed (internal)
constexpr uint32_t kCounters = 36;

struct Open {                                    // a node of the next level: sorted span [a, b] and where it hangs
    uint32_t a, b, parent, side;                 // side 0: parent's left child, 1: its right child
};

struct Bounds { float lo[3], hi[3]; };          // of the finite centroid components; lo = +inf: none on that axis

__device__ __forceinline__ bool finite(float v) { return fabsf(v) <= 3.402823466e38f; }   // false for NaN and +-inf

// The quantisation rule of the header comment, pinned: strict fp32 (strict_math.cuh), no contraction.
__device__ __forceinline__ uint32_t quantise(float c, float lo, float hi) {
    if (c != c || c == __int_as_float(0x7f800000)) return kQuantMax;
    if (c == __int_as_float(0xff800000)) return 0u;
    const float ext = fsub(hi, lo);
    if (!(lo <= hi) || !(finite(ext) && ext > 0.0f)) return 0u;
    const float q = floorf(fmul(fdiv(fsub(c, lo), ext), 2097152.0f));
    return q >= (float)kQuantMax ? kQuantMax : (uint32_t)q;
}

__device__ __forceinline__ uint64_t spread3(uint32_t v) {       // bit i -> bit 3i
    uint64_t x = v & 0x1fffffu;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

// counters zeroed by the caller; bounds start empty; the root opens level 0
__global__ void morton_init_kernel(Bounds* bounds, Open* level0, uint32_t n, uint32_t* counters) {
    if (threadIdx.x != 0) return;
    for (int k = 0; k < 3; ++k) { bounds->lo[k] = __int_as_float(0x7f800000); bounds->hi[k] = __int_as_float(0xff800000); }
    level0[0].a = 0; level0[0].b = n - 1; level0[0].parent = 0; level0[0].side = 0;
    counters[kLevelCounts] = 1;
}

// Bounds of the finite centroid components: warp shuffles, then one atomic per warp and component (min / max are exact,
// so the result does not depend on the order). Non-finite components enter as +inf / -inf, which never win.
__global__ void __launch_bounds__(256)
morton_bounds_kernel(const RefBVH* __restrict__ leaves, uint32_t n, Bounds* bounds) {
    float lo[3], hi[3];
    for (int k = 0; k < 3; ++k) { lo[k] = __int_as_float(0x7f800000); hi[k] = __int_as_float(0xff800000); }
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const f3 c = gpubuild::centroid_of(leaves[i]);
        const float v[3] = {c.x, c.y, c.z};
        for (int k = 0; k < 3; ++k)
            if (finite(v[k])) { lo[k] = fminf(lo[k], v[k]); hi[k] = fmaxf(hi[k], v[k]); }
    }
    for (int off = 16; off > 0; off >>= 1)
        for (int k = 0; k < 3; ++k) {
            lo[k] = fminf(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], off));
            hi[k] = fmaxf(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], off));
        }
    if ((threadIdx.x & 31u) == 0)
        for (int k = 0; k < 3; ++k)
            if (lo[k] <= hi[k]) { gpubuild::atomic_min_f(&bounds->lo[k], lo[k]); gpubuild::atomic_max_f(&bounds->hi[k], hi[k]); }
}

__global__ void __launch_bounds__(256)
morton_code_kernel(const RefBVH* __restrict__ leaves, uint32_t n, const Bounds* __restrict__ bounds, uint64_t* __restrict__ code,
                   uint32_t* __restrict__ pos) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const f3 c = gpubuild::centroid_of(leaves[i]);
    const Bounds b = *bounds;
    code[i] = spread3(quantise(c.x, b.lo[0], b.hi[0])) << 2 | spread3(quantise(c.y, b.lo[1], b.hi[1])) << 1 |
              spread3(quantise(c.z, b.lo[2], b.hi[2]));
    pos[i] = i;
}

// One interior level: every open node of depth `depth` picks its split, is written at its final index, links itself into
// its parent and opens its interior children for the next level. The level's count lives in counters[depth], so the
// launches of all levels are queued back to back.
__global__ void __launch_bounds__(256)
morton_level_kernel(const uint64_t* __restrict__ code, const uint32_t* __restrict__ order, uint32_t n, const Open* __restrict__ cur,
                    Open* __restrict__ next, uint32_t cap, uint32_t* counters, uint32_t depth, RefBVH* out) {
    const uint32_t count = counters[kLevelCounts + depth];
    if (count == 0) return;
    const uint32_t gRoot = depth == 0 ? 0u : counters[kRootGap];
    const uint64_t lim = 1ull << (31 - depth);
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < count; k += gridDim.x * blockDim.x) {
        const Open o = cur[k];
        const uint32_t a = o.a, b = o.b, m = b - a + 1;
        const uint64_t ca = code[a], cb = code[b];
        uint32_t s, axis = 0;
        if (ca == cb) {
            s = m / 2;
        } else {
            const uint32_t h = 63u - (uint32_t)__clzll((long long)(ca ^ cb));
            axis = 2u - h % 3u;
            uint32_t lo = a + 1, hi = b;                // first position with bit h set: code[a] has it clear, code[b] set
            while (lo < hi) {
                const uint32_t mid = lo + (hi - lo) / 2;
                if ((code[mid] >> h) & 1u) hi = mid; else lo = mid + 1;
            }
            s = lo - a;
        }
        if ((uint64_t)s > lim) s = (uint32_t)lim;                                   // depth clamp
        if ((uint64_t)m > lim && (uint64_t)s < (uint64_t)m - lim) s = (uint32_t)((uint64_t)m - lim);
        if (s < 1) s = 1;
        if (s > m - 1) s = m - 1;
        const uint32_t g = a + s - 1;
        uint32_t self = 0;
        if (depth == 0) counters[kRootGap] = g;
        else self = g < gRoot ? n + 1 + g : n + g;

        RefBVH nb;
        nb.parent = o.parent; nb.left = 0; nb.right = 0; nb.axis = axis;
        nb.pType = TRQ_BVH; nb.pIndex = 0; nb.pad[0] = nb.pad[1] = 0;
        nb.bBOX.mini[0] = nb.bBOX.mini[1] = nb.bBOX.mini[2] = FLT_MAX; nb.bBOX.pad0 = 0.0f;       // refit_kernel fills the box
        nb.bBOX.maxi[0] = nb.bBOX.maxi[1] = nb.bBOX.maxi[2] = -FLT_MAX; nb.bBOX.pad1 = 0.0f;
        const uint32_t span[2][2] = {{a, g}, {g + 1, b}};
        for (int c = 0; c < 2; ++c) {
            const uint32_t ca2 = span[c][0], cb2 = span[c][1];
            uint32_t child = 0;
            if (ca2 == cb2) {
                child = 1 + order[ca2];
                out[child].parent = self;
            } else {
                const uint32_t slot = atomicAdd(&counters[kLevelCounts + depth + 1], 1u);
                if (slot < cap && depth + 1 < kMaxLevels) { next[slot].a = ca2; next[slot].b = cb2; next[slot].parent = self; next[slot].side = c; }
                else atomicExch(&counters[kOverflow], 1u);                          // cannot happen (header comment)
            }
            if (c == 0) nb.left = child; else nb.right = child;
        }
        out[self] = nb;
        if (depth > 0) {                                                            // the parent was written one launch earlier
            if (o.side) out[o.parent].right = self; else out[o.parent].left = self;
        }
        atomicMax(&counters[kMaxDepth], depth);
    }
}

}  // namespace morton
}  // namespace trq
