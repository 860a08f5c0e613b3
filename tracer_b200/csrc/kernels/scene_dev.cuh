// tracer_b200/csrc/kernels/scene_dev.cuh -- device-side view of a scene + packed layout encoding.
//
// Data layout in HBM (DESIGN.md section 3):
//   reference arrays, byte-for-byte as uploaded   spheres / squares / cubes / verts / idx / bvh
//   packed interior nodes  64 B = 4 x float4, 64-B aligned, one per interior BVH node, in
//     depth-first order (root = 0):
//       q0 = { left.mini.xyz , bits(leftRef)  }    q1 = { left.maxi.xyz , bits(rightRef) }
//       q2 = { right.mini.xyz, 0 }                 q3 = { right.maxi.xyz, 0 }
//     Both child boxes live in the parent: one 64-B fetch per from-parent step instead of the
//     reference's 12 B of links + two scattered 32-B boxes + 8 B of child type (Render.hh:151-160,211-213).
//   packed triangles: 64-byte records (48 B used = 3 x float4) per triangle LEAF, in depth-first leaf order, so
//     that a test is one 256-bit + one 128-bit request inside one 64-B-aligned record:
//       t0 = { v0.xyz, bits(leafNode) }  t1 = { v1 - v0, 0 }  t2 = { v2 - v0, 0 }  (t3 unused)
//     (the two edge subtractions are the first operations of Triangle::hit_test, Triangle.hh:43-44)
//   packed spheres 32 B = 2 x float4 per sphere LEAF:
//       s0 = { center.xyz, radius }      s1 = { bits(leafNode), bits(pIndex), bits(material), 0 }
//   packed squares 64 B = 4 x float4 per square LEAF (48 B used):
//       q0 = { range_i.x, range_i.y, range_j.x, range_j.y }
//       q1 = { value_k, bits(axis_i | axis_j << 8 | axis_k << 16), bits(material), bits(leafNode) }
//       q2 = { bits(pIndex), 0, 0, 0 }
//   triangle finish records 64 B per triangle LEAF (same slot as the packed triangle), read once per ray that ends on it:
//       n0 = { normal0.xyz, bits(leafNode) }  n1 = { normal1.xyz, bits(pIndex) }  n2 = { normal2.xyz, 0 }
//   Cube leaves are read in place from the 240-byte reference struct (two per Cornell box).
//
// Interior nodes are numbered so that the first `topNodes` of them are the top of the tree in breadth-first order (any
// prefix of that block can be staged in shared memory by the kernel: "index < topCount" is the residency test); the rest
// follow in depth-first order.
//
// Child reference (32 bit): kind in bits 31..29, index in bits 28..0.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../host/layout.h"

namespace trq {

enum : uint32_t {
    REF_INTERIOR = 0u,   // index = packed interior node
    REF_TRI      = 1u,   // index = packed triangle slot
    REF_SPHERE   = 2u,   // index = packed sphere slot
    REF_SQUARE   = 3u,   // index = packed square slot
    REF_CUBE     = 4u,   // index = leaf node in bvhList (reads the reference-layout Cube)
    REF_NOP      = 6u,   // leaf whose pType dispatches to `default: break` (Render.hh:241)
    REF_DONE     = 7u    // traversal finished (never stored in a node)
};
#define TRQ_REF_KIND(r)  ((r) >> 29)
#define TRQ_REF_INDEX(r) ((r) & 0x1fffffffu)
#define TRQ_MAKE_REF(kind, index) (((uint32_t)(kind) << 29) | (uint32_t)(index))
#define TRQ_REF_DONE_WORD 0xffffffffu

struct SceneDev {
    const RefSphere* spheres;
    const RefSquare* squares;
    const RefCube*   cubes;
    const RefVertex* verts;
    const uint32_t*  idx;
    const RefBVH*    bvh;
    const float4*    nodes;     // 4 per interior node
    const float4*    topSoA;    // [4][topStride]: the first topStride interior nodes again, quarter-major (smem staging source)
    uint32_t         topStride;
    const float4*    tris;      // 3 per triangle leaf
    const float4*    sph;       // 2 per sphere leaf
    const float4*    sq;        // 4 per square leaf
    const float4*    triN;      // 4 per triangle leaf (same slot as tris): {n0, leafNode} {n1, pIndex} {n2, 0} {pad}
    uint32_t         rootRef;
    float            rootMin[3], rootMax[3];
    uint32_t         nNode;
};

// Compact per-ray result written by the trace kernels, resolved into trq_hit by resolve_hits.
// Same 32-B footprint as trq_hit so it is resolved in place.
struct CompactHit {
    float    t;
    uint32_t leafNode;   // bvhList index of the winning leaf
    float    u, v;       // triangle barycentrics / cube uv captured at hit time
    uint32_t aux;        // cube / square: front | material << 1; every other hit: bits of ray direction x
    uint32_t hit;        // 0 / 1
    float    dy, dz;     // ray direction y, z (triangle front-face test in resolve_hits without re-reading the ray)
};

// Work-queue head of one trace launch: `head` is the next unclaimed queue slot; `done` counts CTAs that have left the
// kernel. The last CTA to leave zeroes both, so a head of the eager ring is zero between launches (no memset, no resolve
// pass); a launch captured into a CUDA graph zeroes a head of its own instead (trq_api.cu launch_trace).
struct QueueHead {
    unsigned long long head;
    unsigned int       done;
    unsigned int       pad;
};

#define TRQ_GATHER_MAX_RANKS 16
#define TRQ_MAX_PEERS (TRQ_GATHER_MAX_RANKS - 1)

}  // namespace trq
