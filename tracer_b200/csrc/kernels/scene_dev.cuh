// tracer_b200/csrc/kernels/scene_dev.cuh -- device-side view of a scene and the child-reference encoding.
//
// The packed arrays and their record formats: packed_layout.cuh (DESIGN.md section 3).
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
    const float4*    nodes;     // packed arrays (packed_layout.cuh)
    const float4*    topSoA;    // the first topStride interior nodes again, quarter-major (smem staging source)
    uint32_t         topStride;
    const float4*    tris;
    const float4*    sph;
    const float4*    sq;
    const float4*    triN;
    uint32_t         rootRef;
    float            rootMin[3], rootMax[3];
    uint32_t         nNode;
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
