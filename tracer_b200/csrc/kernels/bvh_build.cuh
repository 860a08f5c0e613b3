// tracer_b200/csrc/kernels/bvh_build.cuh -- GPU construction of the reference BVH (SURVEY.md section 8, row f-1).
//
// A level-synchronous, data-parallel evaluation of the reference's top-down binned-SAH builder
// (BVH::make, RT_Metal/Metal/BVH.hh:35-244; buildTree :246-269) that emits the SAME 64-byte node array as the
// sequential host restatement (csrc/host/bvh_build.cpp): same splits, same child order, same node numbering,
// same boxes. What makes that possible:
//   * every quantity that decides a split is an order-independent reduction over the node's primitives:
//     centroid bounds and bucket boxes are min/max (exact, associative), bucket counts are integers, and the
//     SAH costs are then computed per node in the reference's scalar order;
//   * the in-place partition of BVH.hh:152-168 is a Hoare partition: it swaps the k-th misplaced element from
//     the left with the k-th misplaced element from the right and moves nothing else, which prefix sums
//     reproduce exactly (position for position), so even the span-2 / span-1 tie-breaks that look at list order
//     see the list the reference would have;
//   * the sequential builder numbers interior nodes in post-order; a subtree over k leaves creates exactly k-1 of
//     them, so a node's index (N + base + span - 2) and both children's indices are known the moment it is split.
// A node whose centroids all land in bucket 0 takes the sort + median fallback (BVH.hh:187-195): >= 3 primitives on one
// centroid (0/0 in AABB::relative), or centroids spanning an infinite extent on the split axis (a +inf centroid from a
// leaf side at +inf, or centroids near -FLT_MAX and +FLT_MAX: x/inf is 0, inf/inf is NaN). The GPU sorts such a node by
// (key, list position), which is std::sort's one result when the keys are distinct. The documented difference: with
// equal keys std::sort's order is unspecified (the GPU keeps list order), and with a NaN key `<` is no strict weak
// ordering, so the reference's order is not defined at all (the GPU puts NaN after +inf).
#pragma once
#include <cfloat>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../../include/tracer_rq.h"
#include "../host/layout.h"
#include "strict_math.cuh"

namespace trq {
namespace gpubuild {

constexpr uint32_t kBuckets = 10;                // BVH.hh:91
constexpr uint32_t kNone = 0xffffffffu;

struct BNode {                                   // one active subtree (a contiguous range of idx) of the current level
    uint32_t start, end, base;                   // range; interior nodes created before it in post-order
    uint32_t dim, split, mid, fallback, nSwap;
    uint32_t child[2];                           // slots of the children in the next level's table (kNone: leaf / done)
    float cmin[3], cmax[3];                      // bounds of the centroids
    uint32_t bcount[kBuckets];
    float bmin[kBuckets][3], bmax[kBuckets][3];
};

// ---- float atomics on bit patterns (min/max are exact, so the result is order-independent). They agree with the
// host's fminf / fmaxf: a NaN is ignored, and the branch is on the sign BIT, so -0.0 takes the unsigned path
// (v >= 0.0f is true for -0.0, whose bits are INT_MIN as a signed int). -0.0 and +0.0 then order as -0.0 < +0.0,
// which no decision of the builder can see: they are equal in every comparison and give equal areas.
__device__ __forceinline__ void atomic_min_f(float* a, float v) {
    if (v != v) return;
    if (__float_as_int(v) >= 0) atomicMin(reinterpret_cast<int*>(a), __float_as_int(v));
    else                        atomicMax(reinterpret_cast<unsigned int*>(a), __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_f(float* a, float v) {
    if (v != v) return;
    if (__float_as_int(v) >= 0) atomicMax(reinterpret_cast<int*>(a), __float_as_int(v));
    else                        atomicMin(reinterpret_cast<unsigned int*>(a), __float_as_uint(v));
}

// AABB::centroid  AABB.hh:22-25
__device__ __forceinline__ f3 centroid_of(const RefBVH& n) {
    return make_f3(fadd(n.bBOX.mini[0], fdiv(fsub(n.bBOX.maxi[0], n.bBOX.mini[0]), 2.0f)),
                   fadd(n.bBOX.mini[1], fdiv(fsub(n.bBOX.maxi[1], n.bBOX.mini[1]), 2.0f)),
                   fadd(n.bBOX.mini[2], fdiv(fsub(n.bBOX.maxi[2], n.bBOX.mini[2]), 2.0f)));
}
// AABB::maximumExtent  AABB.hh:42-49
__device__ __forceinline__ uint32_t maximum_extent(const float lo[3], const float hi[3]) {
    const float dx = fsub(hi[0], lo[0]), dy = fsub(hi[1], lo[1]), dz = fsub(hi[2], lo[2]);
    if (dx > dy && dx > dz) return 0u;
    return dy > dz ? 1u : 2u;
}
// AABB::area  AABB.hh:27-30
__device__ __forceinline__ float box_area(const float lo[3], const float hi[3]) {
    const float dx = fsub(hi[0], lo[0]), dy = fsub(hi[1], lo[1]), dz = fsub(hi[2], lo[2]);
    return fmul(2.0f, fadd(fadd(fmul(dx, dy), fmul(dx, dz)), fmul(dy, dz)));
}
// bucket of a centroid inside the centroid box  BVH.hh:96-100
__device__ __forceinline__ uint32_t bucket_of(const BNode& nd, float c) {
    const float d = fsub(nd.cmax[nd.dim], nd.cmin[nd.dim]);
    const float scaled = fmul((float)kBuckets, fdiv(fsub(c, nd.cmin[nd.dim]), d));     // nBuckets * relative(centroid)[dim]
    const uint32_t b = (scaled != scaled) ? 0u : (uint32_t)scaled;                     // NaN (all centroids equal) -> 0
    return b < kBuckets - 1 ? b : kBuckets - 1;
}

// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
init_elements_kernel(const RefBVH* __restrict__ leaves, uint32_t n, uint32_t* idx, uint32_t* seg, float4* cen) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    idx[i] = i; seg[i] = 0u;
    const f3 c = centroid_of(leaves[i]);
    cen[i] = make_float4(c.x, c.y, c.z, 0.0f);
}

__global__ void __launch_bounds__(256)
reset_nodes_kernel(BNode* nodes, uint32_t nNodes, uint32_t* nFallback) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *nFallback = 0;
    if (i >= nNodes) return;
    BNode& nd = nodes[i];
    for (int k = 0; k < 3; ++k) { nd.cmin[k] = FLT_MAX; nd.cmax[k] = -FLT_MAX; }       // AABB default (AABB.hh:8-9)
    for (uint32_t b = 0; b < kBuckets; ++b) {
        nd.bcount[b] = 0;
        for (int k = 0; k < 3; ++k) { nd.bmin[b][k] = FLT_MAX; nd.bmax[b][k] = -FLT_MAX; }
    }
    nd.child[0] = nd.child[1] = kNone;
    nd.dim = nd.split = nd.mid = nd.fallback = nd.nSwap = 0;
}

// K1: bounds of the centroids of every active node (BVH.hh:81-87). Warp-uniform segments are reduced with
// shuffles first so that the huge top-level nodes cost n/32 atomics per address, not n.
__global__ void __launch_bounds__(256)
centroid_bounds_kernel(const uint32_t* __restrict__ idx, const uint32_t* __restrict__ seg, const float4* __restrict__ cen,
                       uint32_t n, BNode* nodes) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t s = p < n ? seg[p] : kNone;
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    if (s != kNone) {
        const float4 c = cen[idx[p]];
        lo[0] = hi[0] = c.x; lo[1] = hi[1] = c.y; lo[2] = hi[2] = c.z;
    }
    const uint32_t s0 = __shfl_sync(0xffffffffu, s, 0);
    if (__all_sync(0xffffffffu, s == s0)) {
        if (s0 == kNone) return;
        for (int off = 16; off > 0; off >>= 1)
            for (int k = 0; k < 3; ++k) {
                lo[k] = fminf(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], off));
                hi[k] = fmaxf(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], off));
            }
        if ((threadIdx.x & 31u) == 0)
            for (int k = 0; k < 3; ++k) { atomic_min_f(&nodes[s0].cmin[k], lo[k]); atomic_max_f(&nodes[s0].cmax[k], hi[k]); }
    } else if (s != kNone) {
        for (int k = 0; k < 3; ++k) { atomic_min_f(&nodes[s].cmin[k], lo[k]); atomic_max_f(&nodes[s].cmax[k], hi[k]); }
    }
}

// K2: split axis per node (BVH.hh:69,89)
__global__ void __launch_bounds__(256)
choose_axis_kernel(BNode* nodes, uint32_t nNodes) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nNodes) return;
    nodes[i].dim = maximum_extent(nodes[i].cmin, nodes[i].cmax);
}

// K3: bucket counts and bucket boxes (BVH.hh:94-108). A block whose 256 elements all belong to one node
// accumulates in shared memory and flushes 10 x 7 atomics; mixed blocks (small nodes) go straight to global.
__global__ void __launch_bounds__(256)
bucket_kernel(const RefBVH* __restrict__ leaves, const uint32_t* __restrict__ idx, const uint32_t* __restrict__ seg,
              const float4* __restrict__ cen, uint32_t n, BNode* nodes) {
    __shared__ uint32_t sCount[kBuckets];
    __shared__ float sMin[kBuckets][3], sMax[kBuckets][3];
    __shared__ uint32_t sSeg, sUniform;
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t s = p < n ? seg[p] : kNone;
    if (threadIdx.x == 0) { sSeg = s; sUniform = 1u; }
    if (threadIdx.x < kBuckets) {
        sCount[threadIdx.x] = 0;
        for (int k = 0; k < 3; ++k) { sMin[threadIdx.x][k] = FLT_MAX; sMax[threadIdx.x][k] = -FLT_MAX; }
    }
    __syncthreads();
    if (s != sSeg) sUniform = 0u;                       // benign race: everyone writes the same value
    __syncthreads();
    const bool uniform = sUniform != 0u;
    if (s != kNone) {
        const BNode& nd = nodes[s];
        if (nd.end - nd.start > 2) {                    // span 1 / 2 never reach the bucket code (BVH.hh:52-77)
            const uint32_t leaf = idx[p];
            const float4 c = cen[leaf];
            const uint32_t b = bucket_of(nd, nd.dim == 0 ? c.x : (nd.dim == 1 ? c.y : c.z));
            const RefAABB box = leaves[leaf].bBOX;
            if (uniform) {
                atomicAdd(&sCount[b], 1u);
                for (int k = 0; k < 3; ++k) { atomic_min_f(&sMin[b][k], box.mini[k]); atomic_max_f(&sMax[b][k], box.maxi[k]); }
            } else {
                atomicAdd(&nodes[s].bcount[b], 1u);
                for (int k = 0; k < 3; ++k) { atomic_min_f(&nodes[s].bmin[b][k], box.mini[k]); atomic_max_f(&nodes[s].bmax[b][k], box.maxi[k]); }
            }
        }
    }
    __syncthreads();
    if (uniform && sSeg != kNone && threadIdx.x < kBuckets && sCount[threadIdx.x] > 0) {
        const uint32_t b = threadIdx.x;
        atomicAdd(&nodes[sSeg].bcount[b], sCount[b]);
        for (int k = 0; k < 3; ++k) { atomic_min_f(&nodes[sSeg].bmin[b][k], sMin[b][k]); atomic_max_f(&nodes[sSeg].bmax[b][k], sMax[b][k]); }
    }
}

// K4: SAH cost of the 9 candidate splits in the reference's scalar order and the first strict minimum (BVH.hh:110-139)
__global__ void __launch_bounds__(128)
choose_split_kernel(BNode* nodes, uint32_t nNodes) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nNodes) return;
    BNode& nd = nodes[i];
    if (nd.end - nd.start <= 2) return;
    const float cboxArea = box_area(nd.cmin, nd.cmax);          // area of the CENTROID box, as the reference does
    float cost[kBuckets - 1];
    for (uint32_t s = 0; s < kBuckets - 1; ++s) {
        float lo0[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi0[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
        float lo1[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi1[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
        int count0 = 0, count1 = 0;
        for (uint32_t j = 0; j <= s; ++j) {
            for (int k = 0; k < 3; ++k) { lo0[k] = fminf(lo0[k], nd.bmin[j][k]); hi0[k] = fmaxf(hi0[k], nd.bmax[j][k]); }
            count0 += (int)nd.bcount[j];
        }
        for (uint32_t j = s + 1; j < kBuckets; ++j) {
            for (int k = 0; k < 3; ++k) { lo1[k] = fminf(lo1[k], nd.bmin[j][k]); hi1[k] = fmaxf(hi1[k], nd.bmax[j][k]); }
            count1 += (int)nd.bcount[j];
        }
        cost[s] = fadd(1.0f, fdiv(fadd(fmul((float)count0, box_area(lo0, hi0)), fmul((float)count1, box_area(lo1, hi1))), cboxArea));
    }
    float minCost = cost[0];
    uint32_t best = 0;
    for (uint32_t s = 1; s < kBuckets - 1; ++s)
        if (cost[s] < minCost) { minCost = cost[s]; best = s; }
    nd.split = best;
}

// K5: partition predicate per element (BVH.hh:141-150); 0 outside nodes that partition
__global__ void __launch_bounds__(256)
predicate_kernel(const uint32_t* __restrict__ idx, const uint32_t* __restrict__ seg, const float4* __restrict__ cen,
                 uint32_t n, const BNode* __restrict__ nodes, uint32_t* __restrict__ flag) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p > n) return;
    uint32_t f = 0;
    if (p < n) {
        const uint32_t s = seg[p];
        if (s != kNone) {
            const BNode& nd = nodes[s];
            if (nd.end - nd.start > 2) {
                const float4 c = cen[idx[p]];
                f = bucket_of(nd, nd.dim == 0 ? c.x : (nd.dim == 1 ? c.y : c.z)) <= nd.split ? 1u : 0u;
            }
        }
    }
    flag[p] = f;                                        // flag[n] = 0: the scan then yields a total at [n]
}

// ---- exclusive prefix sum of n uint32 (three passes, 4096 elements per block)
constexpr uint32_t kScanItems = 4;
constexpr uint32_t kScanTile = 1024 * kScanItems;

__global__ void __launch_bounds__(1024)
scan_tiles_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint32_t n, uint32_t* __restrict__ tileSums) {
    __shared__ uint32_t warpSums[32];
    const uint32_t base = blockIdx.x * kScanTile + threadIdx.x * kScanItems;
    uint32_t v[kScanItems], sum = 0;
    for (uint32_t k = 0; k < kScanItems; ++k) { v[k] = (base + k < n) ? in[base + k] : 0u; sum += v[k]; }
    uint32_t incl = sum;
    for (int off = 1; off < 32; off <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, off); if ((threadIdx.x & 31) >= off) incl += t; }
    if ((threadIdx.x & 31) == 31) warpSums[threadIdx.x >> 5] = incl;
    __syncthreads();
    if (threadIdx.x < 32) {
        uint32_t w = warpSums[threadIdx.x];
        for (int off = 1; off < 32; off <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, w, off); if ((int)threadIdx.x >= off) w += t; }
        warpSums[threadIdx.x] = w;
    }
    __syncthreads();
    uint32_t run = incl - sum + ((threadIdx.x >> 5) ? warpSums[(threadIdx.x >> 5) - 1] : 0u);
    for (uint32_t k = 0; k < kScanItems; ++k) { if (base + k < n) out[base + k] = run; run += v[k]; }
    if (threadIdx.x == 1023) tileSums[blockIdx.x] = run;
}

__global__ void __launch_bounds__(1024)
scan_sums_kernel(uint32_t* tileSums, uint32_t nTiles) {        // single block, serial over chunks of 1024 tiles
    __shared__ uint32_t warpSums[32];
    __shared__ uint32_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < nTiles; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = i < nTiles ? tileSums[i] : 0u;
        uint32_t incl = v;
        for (int off = 1; off < 32; off <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, off); if ((threadIdx.x & 31) >= off) incl += t; }
        if ((threadIdx.x & 31) == 31) warpSums[threadIdx.x >> 5] = incl;
        __syncthreads();
        if (threadIdx.x < 32) {
            uint32_t w = warpSums[threadIdx.x];
            for (int off = 1; off < 32; off <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, w, off); if ((int)threadIdx.x >= off) w += t; }
            warpSums[threadIdx.x] = w;
        }
        __syncthreads();
        const uint32_t excl = carry + incl - v + ((threadIdx.x >> 5) ? warpSums[(threadIdx.x >> 5) - 1] : 0u);
        if (i < nTiles) tileSums[i] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) carry = excl + v;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(1024)
scan_add_kernel(uint32_t* __restrict__ out, uint32_t n, const uint32_t* __restrict__ tileSums) {
    const uint32_t base = blockIdx.x * kScanTile + threadIdx.x * kScanItems;
    const uint32_t add = tileSums[blockIdx.x];
    for (uint32_t k = 0; k < kScanItems; ++k) if (base + k < n) out[base + k] += add;
}

// K6: partition point per node, fallback detection (BVH.hh:187-195), number of Hoare swaps
__global__ void __launch_bounds__(256)
midpoint_kernel(BNode* nodes, uint32_t nNodes, const uint32_t* __restrict__ scanT, uint32_t* fallbackList, uint32_t* nFallback) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nNodes) return;
    BNode& nd = nodes[i];
    const uint32_t span = nd.end - nd.start;
    if (span <= 2) return;
    const uint32_t nT = scanT[nd.end] - scanT[nd.start];
    uint32_t mid = nd.start + nT;
    nd.fallback = 0; nd.nSwap = 0;
    if (mid <= nd.start || mid >= nd.end) {             // every centroid in one bucket set: sort + median split in the reference
        nd.fallback = 1;
        mid = nd.start + span / 2;
        fallbackList[atomicAdd(nFallback, 1u)] = i;
    } else {
        nd.nSwap = (mid - nd.start) - (scanT[mid] - scanT[nd.start]);     // misplaced (false) elements left of mid
    }
    nd.mid = mid;
}

// K7: list the misplaced elements: k-th false from the left, k-th true from the right (BVH.hh:152-168)
__global__ void __launch_bounds__(256)
mispl_kernel(const uint32_t* __restrict__ seg, uint32_t n, const BNode* __restrict__ nodes, const uint32_t* __restrict__ flag,
             const uint32_t* __restrict__ scanT, uint32_t* __restrict__ leftFalse, uint32_t* __restrict__ rightTrue) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const uint32_t s = seg[p];
    if (s == kNone) return;
    const BNode& nd = nodes[s];
    if (nd.end - nd.start <= 2 || nd.fallback) return;
    if (p < nd.mid) {
        if (!flag[p]) leftFalse[nd.start + ((p - nd.start) - (scanT[p] - scanT[nd.start]))] = p;
    } else {
        if (flag[p]) rightTrue[nd.start + (scanT[nd.end] - scanT[p + 1])] = p;
    }
}

// K8: perform the swaps
__global__ void __launch_bounds__(256)
swap_kernel(const uint32_t* __restrict__ seg, uint32_t n, const BNode* __restrict__ nodes,
            const uint32_t* __restrict__ leftFalse, const uint32_t* __restrict__ rightTrue, uint32_t* idx) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    const uint32_t s = seg[q];
    if (s == kNone) return;
    const BNode& nd = nodes[s];
    if (q - nd.start >= nd.nSwap) return;
    const uint32_t a = leftFalse[q], b = rightTrue[q];
    const uint32_t ia = idx[a], ib = idx[b];
    idx[a] = ib; idx[b] = ia;
}

// K8b: the fallback's std::sort of the node's idx range by centroid[dim] (BVH.hh:187-195), one block per listed node.
// Keys are (order-preserving bits of the centroid, position in the range): all distinct, so the result is the stable
// sort. The network is bitonic with every comparator sending the smaller key to the lower index (the first step of each
// merge pairs mirrored positions): positions past the span act as +inf padding that no comparator moves, so the
// range is sorted in place in the 64-bit scratch `keys` (indexed by list position, like idx).
constexpr uint32_t kSortThreads = 512;
constexpr uint32_t kSortBlocks = 256;

__device__ __forceinline__ uint32_t sort_bits(float f) {       // -0.0 -> +0.0 first: they are equal under `<`
    const uint32_t u = __float_as_uint(f == 0.0f ? 0.0f : f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__global__ void __launch_bounds__(kSortThreads)
fallback_sort_kernel(const BNode* __restrict__ nodes, const uint32_t* __restrict__ fallbackList, const uint32_t* __restrict__ nFallback,
                     const float4* __restrict__ cen, uint32_t* idx, unsigned long long* keys) {
    const uint32_t count = *nFallback;
    for (uint32_t f = blockIdx.x; f < count; f += gridDim.x) {
        const BNode& nd = nodes[fallbackList[f]];
        const uint32_t start = nd.start, span = nd.end - nd.start, dim = nd.dim;
        unsigned long long* k = keys + start;
        for (uint32_t t = threadIdx.x; t < span; t += blockDim.x) {
            const float4 c = cen[idx[start + t]];
            k[t] = ((unsigned long long)sort_bits(dim == 0 ? c.x : (dim == 1 ? c.y : c.z)) << 32) | t;
        }
        __syncthreads();
        uint32_t pow2 = 1;
        while (pow2 < span) pow2 <<= 1;
        for (uint32_t size = 2; size <= pow2; size <<= 1)
            for (uint32_t j = size >> 1; j > 0; j >>= 1) {
                for (uint32_t t = threadIdx.x; t < pow2 / 2; t += blockDim.x) {
                    const uint32_t lo = 2 * (t & ~(j - 1)) + (t & (j - 1));
                    const uint32_t hi = j == size >> 1 ? lo ^ (size - 1) : lo + j;
                    if (hi < span) {
                        const unsigned long long a = k[lo], b = k[hi];
                        if (b < a) { k[lo] = b; k[hi] = a; }
                    }
                }
                __syncthreads();
            }
        for (uint32_t t = threadIdx.x; t < span; t += blockDim.x) k[t] = idx[start + (uint32_t)k[t]];
        __syncthreads();
        for (uint32_t t = threadIdx.x; t < span; t += blockDim.x) idx[start + t] = (uint32_t)k[t];
        __syncthreads();
    }
}

// K9: emit the interior node of every active subtree and open its children for the next level (BVH.hh:222-243)
__global__ void __launch_bounds__(128)
emit_kernel(BNode* nodes, uint32_t nNodes, const uint32_t* __restrict__ idx, const float4* __restrict__ cen,
            RefBVH* out /* final layout: root at 0, pre-shift index j at j+1 */, uint32_t nLeaves,
            BNode* next, uint32_t cap /* entries of `next` */, uint32_t* nNext, uint32_t* overflow, uint32_t* maxDepth, uint32_t depth) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nNodes) return;
    BNode& nd = nodes[i];
    const uint32_t span = nd.end - nd.start;
    const uint32_t self = nLeaves + nd.base + span - 2;             // pre-shift index == bvh_list.size() at emplace time
    const uint32_t selfFinal = (self == 2 * nLeaves - 2) ? 0u : self + 1;
    uint32_t childPre[2];                                           // pre-shift indices of left / right
    uint32_t dim;
    if (span == 2) {                                                // BVH.hh:60-77
        const uint32_t ia = idx[nd.start], ib = idx[nd.start + 1];
        const float4 ca = cen[ia], cb = cen[ib];
        // AABB::make(a, b) grows the default box (AABB.hh:8-9): a component that is NaN in both centroids stays
        // (FLT_MAX, -FLT_MAX), an extent of -inf rather than NaN, and maximumExtent sees the difference
        const float lo[3] = {fminf(fminf(FLT_MAX, ca.x), cb.x), fminf(fminf(FLT_MAX, ca.y), cb.y), fminf(fminf(FLT_MAX, ca.z), cb.z)};
        const float hi[3] = {fmaxf(fmaxf(-FLT_MAX, ca.x), cb.x), fmaxf(fmaxf(-FLT_MAX, ca.y), cb.y), fmaxf(fmaxf(-FLT_MAX, ca.z), cb.z)};
        dim = maximum_extent(lo, hi);
        const float ka = dim == 0 ? ca.x : (dim == 1 ? ca.y : ca.z), kb = dim == 0 ? cb.x : (dim == 1 ? cb.y : cb.z);
        if (ka < kb) { childPre[0] = ia; childPre[1] = ib; } else { childPre[0] = ib; childPre[1] = ia; }
    } else {
        dim = nd.dim;
        const uint32_t lspan = nd.mid - nd.start, rspan = nd.end - nd.mid;
        const uint32_t lbase = nd.base, rbase = nd.base + (lspan - 1);
        childPre[0] = lspan == 1 ? idx[nd.start] : nLeaves + lbase + lspan - 2;
        childPre[1] = rspan == 1 ? idx[nd.mid] : nLeaves + rbase + rspan - 2;
        if (lspan > 1) {
            const uint32_t slot = atomicAdd(nNext, 1u);
            if (slot < cap) { next[slot].start = nd.start; next[slot].end = nd.mid; next[slot].base = lbase; nd.child[0] = slot; }
            else atomicExch(overflow, 1u);                          // cannot happen (a level has at most n/2 open subtrees); never write past the table
        }
        if (rspan > 1) {
            const uint32_t slot = atomicAdd(nNext, 1u);
            if (slot < cap) { next[slot].start = nd.mid; next[slot].end = nd.end; next[slot].base = rbase; nd.child[1] = slot; }
            else atomicExch(overflow, 1u);
        }
        atomicMax(maxDepth, depth);
    }
    if (span == 2) atomicMax(maxDepth, depth);
    RefBVH nb;
    nb.parent = 0; nb.axis = dim;
    nb.left = childPre[0] + 1; nb.right = childPre[1] + 1;          // BVH.hh:225-226 (final indices)
    nb.pType = TRQ_BVH; nb.pIndex = 0; nb.pad[0] = nb.pad[1] = 0;
    // box = union of the two child boxes (BVH.hh:229-231) = union of every leaf box below (min/max are exact);
    // filled in by the bottom-up pass (refit_kernel) once the children exist.
    nb.bBOX.mini[0] = nb.bBOX.mini[1] = nb.bBOX.mini[2] = FLT_MAX; nb.bBOX.pad0 = 0.0f;
    nb.bBOX.maxi[0] = nb.bBOX.maxi[1] = nb.bBOX.maxi[2] = -FLT_MAX; nb.bBOX.pad1 = 0.0f;
    // parent links of the children (BVH.hh:240-241); this node's own parent is written by ITS parent
    const uint32_t keepParent = out[selfFinal].parent;              // may already have been set by the parent (previous level)
    nb.parent = keepParent;
    out[selfFinal] = nb;
    out[childPre[0] + 1].parent = selfFinal;
    out[childPre[1] + 1].parent = selfFinal;
}

// K10: move every element to its child's slot in the next level's table
__global__ void __launch_bounds__(256)
reseg_kernel(uint32_t* seg, uint32_t n, const BNode* __restrict__ nodes) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const uint32_t s = seg[p];
    if (s == kNone) return;
    const BNode& nd = nodes[s];
    seg[p] = (nd.end - nd.start == 2) ? kNone : nd.child[p < nd.mid ? 0 : 1];
}

// Bottom-up boxes: interior pre-shift indices are in post-order, so children always have SMALLER indices than
// their parent; processing interior nodes level by level from the deepest is not needed -- one thread per leaf
// climbs to the root, the second arrival at a node (atomic counter) merges the two child boxes. (Karras-style.)
__global__ void __launch_bounds__(256)
refit_kernel(RefBVH* out, uint32_t nLeaves, uint32_t* arrivals) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nLeaves || nLeaves < 2) return;
    uint32_t node = out[1 + i].parent;                              // leaves live at 1..nLeaves
    for (;;) {
        if (atomicAdd(&arrivals[node], 1u) == 0u) return;           // first child to arrive waits for its sibling
        __threadfence();
        const RefBVH* l = &out[out[node].left];
        const RefBVH* r = &out[out[node].right];
        for (int k = 0; k < 3; ++k) {                               // __ldcg: child boxes were written by other SMs in this launch
            out[node].bBOX.mini[k] = fminf(__ldcg(&l->bBOX.mini[k]), __ldcg(&r->bBOX.mini[k]));   // AABB::make(box, box)  AABB.hh:227-239
            out[node].bBOX.maxi[k] = fmaxf(__ldcg(&l->bBOX.maxi[k]), __ldcg(&r->bBOX.maxi[k]));
        }
        __threadfence();
        if (node == 0) return;
        node = out[node].parent;
    }
}

}  // namespace gpubuild
}  // namespace trq
