// tracer_b200/csrc/kernels/packed_layout.cuh -- the packed traversal layout: record formats, array sizes, the writer
// (pack_scene_kernel) and the readers the trace kernel uses. Nothing else derives a packed address or size.
//
// Data layout in HBM (DESIGN.md section 3):
//   reference arrays, byte-for-byte as uploaded   spheres / squares / cubes / verts / idx / bvh
//   packed interior nodes  64 B = 4 x float4, 64-B aligned, one per interior BVH node (root = 0):
//       q0 = { left.mini.xyz , bits(leftRef)  }    q1 = { left.maxi.xyz , bits(rightRef) }
//       q2 = { right.mini.xyz, 0 }                 q3 = { right.maxi.xyz, 0 }
//     Both child boxes live in the parent: one 64-B fetch per from-parent step instead of the
//     reference's 12 B of links + two scattered 32-B boxes + 8 B of child type (Render.hh:151-160,211-213).
//     The first `topNodes` (at most kTopMax) are the top of the tree in breadth-first order (any prefix of that block can be
//     staged in shared memory by the kernel: "index < topCount" is the residency test); the rest follow in depth-first order.
//   top-of-tree block: the first `topNodes` interior nodes again, quarter-major ([4][topNodes] float4: all q0, then all q1,
//     ...), the source of the staging copy. With the node-major 64-byte stride every q0 would sit in banks 0-3 / 16-19 and a
//     warp's LDS.128 would serialise 4 ways.
//   packed triangles: 64-byte records (48 B used = 3 x float4) per triangle LEAF, in depth-first leaf order, so
//     that a test is one 256-bit + one 128-bit request inside one 64-B-aligned record:
//       t0 = { v0.xyz, bits(leafNode) }  t1 = { v1 - v0, 0 }  t2 = { v2 - v0, 0 }  (t3 unused)
//     (the two edge subtractions are the first operations of Triangle::hit_test, Triangle.hh:43-44)
//   triangle finish records 64 B per triangle LEAF (same slot as the packed triangle), read once per ray that ends on it:
//       n0 = { normal0.xyz, bits(leafNode) }  n1 = { normal1.xyz, bits(pIndex) }  n2 = { normal2.xyz, 0 }  n3 = 0
//   packed spheres 32 B = 2 x float4 per sphere LEAF:
//       s0 = { center.xyz, radius }      s1 = { bits(leafNode), bits(pIndex), bits(material), 0 }
//   packed squares 64 B = 4 x float4 per square LEAF (48 B used):
//       q0 = { range_i.x, range_i.y, range_j.x, range_j.y }
//       q1 = { value_k, bits(axis_i | axis_j << 8 | axis_k << 16), bits(material), bits(leafNode) }
//       q2 = { bits(pIndex), 0, 0, 0 }  q3 = 0
//   Cube leaves are read in place from the 240-byte reference struct (two per Cornell box).
//
// Child references (kind in bits 31..29, index in bits 28..0) are defined in scene_dev.cuh.
#pragma once
#include "intersect.cuh"
#include "scene_dev.cuh"

namespace trq {

__device__ __forceinline__ float4 ldg4(const float4* p) { return __ldg(p); }

// 256-bit read-only load (LDG.E.256 on sm_100): two float4 from a 32-byte aligned address.
__device__ __forceinline__ void ldg8(const float4* p, float4& a, float4& b) {
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "l"(p));
}

namespace packed {

constexpr uint32_t kTopMax = 2047;         // interior nodes numbered breadth-first at the front (11 full levels)
constexpr uint32_t kNodeF4 = 4, kTriF4 = 4, kTriFinishF4 = 4, kSphereF4 = 2, kSquareF4 = 4;   // float4 per record
constexpr size_t kNodeBytes = kNodeF4 * sizeof(float4);    // per interior node, in HBM and staged in shared memory

// Bytes of each packed array for these counts of interior nodes, triangle / sphere / square leaves and top-block nodes
struct Sizes { size_t nodes, tris, triN, sph, sq, top; };
__host__ __device__ inline Sizes sizes(uint32_t nInterior, uint32_t nTri, uint32_t nSphere, uint32_t nSquare, uint32_t topNodes) {
    constexpr size_t f4 = sizeof(float4);
    return {nInterior * kNodeBytes, nTri * (kTriF4 * f4), nTri * (kTriFinishF4 * f4), nSphere * (kSphereF4 * f4), nSquare * (kSquareF4 * f4),
            topNodes * kNodeBytes};
}
__device__ __forceinline__ uint32_t staged_words(uint32_t topCount) { return topCount * (kNodeF4 * 4u); }   // shared-memory words

// readers: an interior node from global memory (two 256-bit requests) or from the staged top block ([4][topCount] float4 in
// shared memory: four LDS.128)
__device__ __forceinline__ void load_node(const float4* nodes, uint32_t ni, float4& q0, float4& q1, float4& q2, float4& q3) {
    const float4* np = nodes + (size_t)ni * kNodeF4;
    ldg8(np, q0, q1); ldg8(np + 2, q2, q3);
}
__device__ __forceinline__ void load_staged_node(const float4* top, uint32_t topCount, uint32_t ni, float4& q0, float4& q1, float4& q2, float4& q3) {
    const float4* tp = top + ni;
    q0 = tp[0]; q1 = tp[topCount]; q2 = tp[2u * topCount]; q3 = tp[3u * topCount];
}

// Top-of-tree staging: TMA bulk copies (cp.async.bulk, completion on an mbarrier) bring the first `count` nodes of the
// quarter-major top block (row stride srcStride) into shared memory ([4][count] float4) when the CTA starts.
__device__ __forceinline__ void stage_top_of_tree(float4* dst, const float4* src, uint32_t count, uint32_t srcStride, unsigned long long* mbar) {
    const uint32_t mb = (uint32_t)__cvta_generic_to_shared(mbar);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(mb));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (count == 0) return;
    if (threadIdx.x == 0) {
        const uint32_t bytes = count * 16u;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mb), "r"(4u * bytes) : "memory");
#pragma unroll
        for (uint32_t q = 0; q < 4; ++q)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         :: "r"((uint32_t)__cvta_generic_to_shared(dst + (size_t)q * count)), "l"(src + (size_t)q * srcStride), "r"(bytes), "r"(mb) : "memory");
    }
    uint32_t ready = 0;
    while (!ready) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ready) : "r"(mb) : "memory");
    }
}

// the used 48 bytes of a 64-byte record (triangle test, triangle finish, square finish): one 256-bit + one 128-bit request
__device__ __forceinline__ void load48(const float4* p, float4& a, float4& b, float4& c) { ldg8(p, a, b); c = ldg4(p + 2); }
__device__ __forceinline__ void load_tri(const float4* tris, uint32_t slot, float4& t0, float4& t1, float4& t2) { load48(tris + (size_t)slot * kTriF4, t0, t1, t2); }
__device__ __forceinline__ void load_tri_finish(const float4* triN, uint32_t slot, float4& n0, float4& n1, float4& n2) {
    load48(triN + (size_t)slot * kTriFinishF4, n0, n1, n2);
}
// a sphere: the test reads s0, the finish the whole record
__device__ __forceinline__ float4 load_sphere_test(const float4* sph, uint32_t slot) { return ldg4(sph + (size_t)slot * kSphereF4); }
__device__ __forceinline__ void load_sphere(const float4* sph, uint32_t slot, float4& s0, float4& s1) {
    s0 = ldg4(sph + (size_t)slot * kSphereF4); s1 = ldg4(sph + (size_t)slot * kSphereF4 + 1);
}
// a square: the test reads q0, q1 (one 256-bit request), the finish the used part of the record
__device__ __forceinline__ void load_square_test(const float4* sq, uint32_t slot, float4& q0, float4& q1) { ldg8(sq + (size_t)slot * kSquareF4, q0, q1); }
__device__ __forceinline__ void load_square(const float4* sq, uint32_t slot, float4& q0, float4& q1, float4& q2) { load48(sq + (size_t)slot * kSquareF4, q0, q1, q2); }

// writers, one per record kind
__device__ __forceinline__ void write_node(float4* nodes, float4* topSoA, uint32_t topStride, uint32_t slot,
                                           const RefAABB& lb, const RefAABB& rb, uint32_t lref, uint32_t rref) {
    const float4 q[4] = {make_float4(lb.mini[0], lb.mini[1], lb.mini[2], __uint_as_float(lref)),
                         make_float4(lb.maxi[0], lb.maxi[1], lb.maxi[2], __uint_as_float(rref)),
                         make_float4(rb.mini[0], rb.mini[1], rb.mini[2], 0.0f),
                         make_float4(rb.maxi[0], rb.maxi[1], rb.maxi[2], 0.0f)};
#pragma unroll
    for (uint32_t k = 0; k < 4; ++k) {
        nodes[(size_t)slot * kNodeF4 + k] = q[k];
        if (slot < topStride) topSoA[(size_t)k * topStride + slot] = q[k];   // a node of the top block: its quarter-major copy too
    }
}
__device__ __forceinline__ void write_tri(float4* tris, uint32_t slot, uint32_t leafNode, const f3& v0, const f3& v1, const f3& v2) {
    const f3 e1 = sub3(v1, v0), e2 = sub3(v2, v0);             // Triangle.hh:43-44
    float4* out = tris + (size_t)slot * kTriF4;
    out[0] = make_float4(v0.x, v0.y, v0.z, __uint_as_float(leafNode));
    out[1] = make_float4(e1.x, e1.y, e1.z, 0.0f);
    out[2] = make_float4(e2.x, e2.y, e2.z, 0.0f);
}
// what a finished triangle hit needs beyond (t, u, v): the vertex normals for checkFace, and its ids
__device__ __forceinline__ void write_tri_finish(float4* triN, uint32_t slot, uint32_t leafNode, uint32_t pIndex,
                                                 const f3& n0, const f3& n1, const f3& n2) {
    float4* out = triN + (size_t)slot * kTriFinishF4;
    out[0] = make_float4(n0.x, n0.y, n0.z, __uint_as_float(leafNode));
    out[1] = make_float4(n1.x, n1.y, n1.z, __uint_as_float(pIndex));
    out[2] = make_float4(n2.x, n2.y, n2.z, 0.0f);
    out[3] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
}
__device__ __forceinline__ void write_sphere(float4* sph, uint32_t slot, uint32_t leafNode, uint32_t pIndex, const RefSphere& s) {
    float4* out = sph + (size_t)slot * kSphereF4;
    out[0] = make_float4(s.center[0], s.center[1], s.center[2], s.radius);
    out[1] = make_float4(__uint_as_float(leafNode), __uint_as_float(pIndex), __uint_as_float(s.material), 0.0f);
}
__device__ __forceinline__ void write_square(float4* sq, uint32_t slot, uint32_t leafNode, uint32_t pIndex, const RefSquare& q) {
    float4* out = sq + (size_t)slot * kSquareF4;
    const uint32_t axes = (uint32_t)q.axis_i | ((uint32_t)q.axis_j << 8) | ((uint32_t)q.axis_k << 16);
    out[0] = make_float4(q.range_i[0], q.range_i[1], q.range_j[0], q.range_j[1]);
    out[1] = make_float4(q.value_k, __uint_as_float(axes), __uint_as_float(q.material), __uint_as_float(leafNode));
    out[2] = make_float4(__uint_as_float(pIndex), 0.0f, 0.0f, 0.0f);
    out[3] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
}

}  // namespace packed

// Derives the packed layout from the reference-layout buffers, one thread per BVH node.
__global__ void __launch_bounds__(256)
pack_scene_kernel(const RefBVH* __restrict__ bvh, const uint32_t* __restrict__ ref, uint32_t nNode,
                  const RefVertex* __restrict__ verts, const uint32_t* __restrict__ idx,
                  const RefSphere* __restrict__ spheres, const RefSquare* __restrict__ squares,
                  float4* __restrict__ nodes, float4* __restrict__ tris, float4* __restrict__ sph, float4* __restrict__ sq,
                  float4* __restrict__ triN, float4* __restrict__ topSoA, uint32_t topStride) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nNode) return;
    const uint32_t my = ref[i];
    const uint32_t kind = TRQ_REF_KIND(my), slot = TRQ_REF_INDEX(my);
    if (my == TRQ_REF_DONE_WORD) return;                      // unreachable node
    if (kind == REF_INTERIOR) {
        const uint32_t l = bvh[i].left, r = bvh[i].right;
        packed::write_node(nodes, topSoA, topStride, slot, bvh[l].bBOX, bvh[r].bBOX, ref[l], ref[r]);
    } else if (kind == REF_TRI) {
        const uint32_t p = bvh[i].pIndex;
        const RefVertex &a = verts[idx[3 * p]], &b = verts[idx[3 * p + 1]], &c = verts[idx[3 * p + 2]];
        packed::write_tri(tris, slot, i, ld3(a.v), ld3(b.v), ld3(c.v));
        packed::write_tri_finish(triN, slot, i, p, ld3(a.n), ld3(b.n), ld3(c.n));
    } else if (kind == REF_SPHERE) {
        packed::write_sphere(sph, slot, i, bvh[i].pIndex, spheres[bvh[i].pIndex]);
    } else if (kind == REF_SQUARE) {
        packed::write_square(sq, slot, i, bvh[i].pIndex, squares[bvh[i].pIndex]);
    }
}

}  // namespace trq
