// tracer_b200/csrc/kernels/trace_kernels.cuh -- the ray-query kernels (sm_100a).
//
//   trace_reflayout_kernel  1:1 transcription of Scene::hit (Render.hh:135-252) over the reference-
//                           layout buffers: parent links + 32-bit trail, one thread per ray.
//                           Correctness anchor and naive baseline (followed by resolve_hits_kernel).
//   trace_packed_kernel     the product kernel: persistent warps pull rays from a global queue with
//                           one warp-aggregated atomic per refill, traverse the packed 64-B fused
//                           nodes with 256-bit loads (the top levels optionally from a TMA-staged copy in
//                           shared memory), and keep the far children of "both hit" nodes
//                           on a per-lane shared-memory stack. The stack replaces the reference's
//                           from-child steps (re-reading parent links, Render.hh:189-209); the visit
//                           ORDER per ray is exactly the reference's: near child first by hit_t's t,
//                           ties to the right child, the far child decided at first arrival and never
//                           re-tested, including the "select the missed child" quirk of Render.hh:174.
//                           A retiring ray's FINAL record (trq_hit, or the 16-byte trq_hit16) is written by
//                           this kernel for every leaf type -- there is no second pass over the batch. One
//                           instance per set of leaf types a tree can have (LEAVES), so that a mesh scene
//                           carries no Sphere / Square / Cube code. Under trq_trace_gather it also counts the
//                           finished records of every tile, for:
//   gather_send_tma_kernel  the collective half of trq_trace_gather: resident BESIDE the trace kernel, ships each
//                           complete tile of records to every peer GPU with TMA bulk copies over NVLink peer
//                           memory while the traversal is still running (gather_send_kernel: the LSU fallback)
//   sort_*_kernel           optional ordering of the work queue (TRQ_SORT_RAYS)
//   expand_hits_kernel      trq_hit -> HitRecord fields (p, gn, sn, uv, f, material)
#pragma once
#include <cfloat>

#include "../../../include/tracer_rq.h"
#include "intersect.cuh"
#include "packed_layout.cuh"
#include "scene_dev.cuh"

namespace trq {

// Batch size of a launch: `n` from the host, or -- for trq_trace_indirect, where the count was produced on the
// device by a spawn kernel -- *nPtr clamped to the capacity n.
__device__ __forceinline__ uint64_t live_count(uint64_t n, const unsigned long long* nPtr) {
    if (nPtr == nullptr) return n;
    const unsigned long long m = *nPtr;
    return m < n ? (uint64_t)m : n;
}

// 256-bit store (STG.E.256 on sm_100): one request for a whole 32-byte record.
__device__ __forceinline__ void stg8(void* p, const float4& a, const float4& b) {
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "l"(p), "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w), "f"(b.x), "f"(b.y), "f"(b.z), "f"(b.w) : "memory");
}

// aux: cube hits = front | material << 1; every other hit = bits of the ray direction's x, with y and z in dy / dz,
// so that resolve_hits_kernel can do a triangle's front-face test without reading the ray again.
__device__ __forceinline__ void store_compact(trq_hit* hits, uint64_t i, bool hit, float t, uint32_t leaf,
                                              float u, float v, uint32_t aux, float dy = 0.0f, float dz = 0.0f) {
    float4 a, b;
    a.x = hit ? t : 0.0f;
    a.y = __uint_as_float(hit ? leaf : 0u);
    a.z = hit ? u : 0.0f;
    a.w = hit ? v : 0.0f;
    b.x = __uint_as_float(hit ? aux : 0u);
    b.y = __uint_as_float(hit ? 1u : 0u);
    b.z = dy; b.w = dz;
    stg8(hits + i, a, b);
}

// Leaf tests that read reference-layout structs (rare leaf types: Square, Cube). Out of line and fed with
// scalars by value so that the hot loops keep the ray in registers (no local-memory RayCtx); the ray context is
// rebuilt here (1/d recomputed: same bits). out = {t, u, v, bits(aux)}. Returns true on accept.
__device__ __noinline__ bool leaf_square_cube(const RefBVH* __restrict__ bvh, const RefSquare* __restrict__ squares,
                                              const RefCube* __restrict__ cubes, uint32_t kind, uint32_t leafNode,
                                              float ox, float oy, float oz, float dx, float dy, float dz,
                                              float range_y, float4* out) {
    const RayCtx ray = make_ray_ctx(ox, oy, oz, dx, dy, dz);
    const uint32_t pIndex = bvh[leafNode].pIndex;
    float t = 0.0f;
    if (kind == REF_SQUARE) {
        if (!square_hit(&squares[pIndex], ray, FLT_MIN, range_y, t, nullptr)) return false;
        *out = make_float4(t, 0.0f, 0.0f, 0.0f);
        return true;
    }
    Surface s;
    if (!cube_hit(&cubes[pIndex], ray, FLT_MIN, range_y, t, &s)) return false;
    *out = make_float4(t, s.uvx, s.uvy, __uint_as_float(s.front | (s.material << 1)));
    return true;
}

// ---------------------------------------------------------------------------------------------
// v0: reference layout, reference control flow.
template <bool ANY>
__global__ void __launch_bounds__(128)
trace_reflayout_kernel(SceneDev S, const trq_ray* __restrict__ rays, trq_hit* __restrict__ hits, uint64_t n,
                       const unsigned long long* __restrict__ nPtr) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= live_count(n, nPtr)) return;
    const float4 r0 = ldg4(reinterpret_cast<const float4*>(rays + i));
    const float4 r1 = ldg4(reinterpret_cast<const float4*>(rays + i) + 1);
    const RayCtx ray = make_ray_ctx(r0.x, r0.y, r0.z, r1.x, r1.y, r1.z);
    const float test_t = r0.w;
    const RefBVH* __restrict__ N = S.bvh;

    uint32_t the_index = 0, tested_index = 0xffffffffu;                   // Render.hh:137-138
    uint32_t stack_mark = 0, stack_level = 0;                             // :140-141
    float range_y = test_t;                                               // :143  range_t = (FLT_MIN, test_t)
    uint32_t best = 0xffffffffu, aux = 0; float bu = 0.0f, bv = 0.0f;
    bool done_any = false;

    if (box_hit(ld3(N[0].bBOX.mini), ld3(N[0].bBOX.maxi), ray, FLT_MIN, range_y)) {   // :145
        do {
            uint32_t sel;
            const uint4 links = *reinterpret_cast<const uint4*>(&N[the_index]);       // parent,left,right,axis :151-153
            const uint32_t p = links.x, l = links.y, r = links.z;
            if (tested_index != l && tested_index != r) {                 // :155
                float tl = range_y, tr = range_y;                         // :157
                const bool lt = box_hit_t(ld3(N[l].bBOX.mini), ld3(N[l].bBOX.maxi), ray, FLT_MIN, range_y, tl);   // :159
                const bool rt = box_hit_t(ld3(N[r].bBOX.mini), ld3(N[r].bBOX.maxi), ray, FLT_MIN, range_y, tr);   // :160
                if (!lt && !rt) { tested_index = the_index; the_index = p; stack_level -= 1; continue; }          // :162-169
                if (lt && rt) stack_mark |= 1u << (stack_level & 31u);    // :171-172
                sel = (tl < tr) ? l : r;                                  // :174
            } else {
                const uint32_t need = (stack_mark >> (stack_level & 31u)) & 1u;       // :191
                stack_mark &= ~(1u << (stack_level & 31u));               // :193
                if (need == 0) { tested_index = the_index; the_index = p; stack_level -= 1; continue; }           // :195-202
                sel = (tested_index == l) ? r : l;                        // :204-208
            }
            const int32_t pType = N[sel].pType;                           // :211-213
            const uint32_t pIndex = N[sel].pIndex;
            bool h = false; float t = 0.0f, u = 0.0f, v = 0.0f; uint32_t a = 0;
            if (pType == TRQ_BVH) { the_index = sel; stack_level += 1; continue; }    // :215-220
            if (pType == TRQ_TRIANGLE) {                                  // :230-240
                const f3 v0 = ld3(S.verts[S.idx[3 * pIndex]].v);
                const f3 v1 = ld3(S.verts[S.idx[3 * pIndex + 1]].v);
                const f3 v2 = ld3(S.verts[S.idx[3 * pIndex + 2]].v);
                h = tri_hit(v0, sub3(v1, v0), sub3(v2, v0), ray, FLT_MIN, range_y, t, u, v);
            } else if (pType == TRQ_SPHERE) {                             // :221-223
                h = sphere_hit(ld3(S.spheres[pIndex].center), S.spheres[pIndex].radius, ray, FLT_MIN, range_y, t);
            } else if (pType == TRQ_SQUARE || pType == TRQ_CUBE) {        // :224-229
                float4 o4;
                h = leaf_square_cube(S.bvh, S.squares, S.cubes, pType == TRQ_SQUARE ? REF_SQUARE : REF_CUBE, sel,
                                     ray.o.x, ray.o.y, ray.o.z, ray.d.x, ray.d.y, ray.d.z, range_y, &o4);
                if (h) { t = o4.x; u = o4.y; v = o4.z; a = __float_as_uint(o4.w); }
            }
            if (h) {                                                      // aux word: cube front/material, else d.x (see store_compact)
                range_y = t; best = sel; bu = u; bv = v;
                aux = (pType == TRQ_SQUARE || pType == TRQ_CUBE) ? a : __float_as_uint(ray.d.x);
            }
            if (ANY && range_y < test_t) { done_any = true; break; }      // :244
            tested_index = sel;                                           // :246
        } while (tested_index != 0);                                      // :248
    }
    const bool hit = done_any || (range_y < test_t);                      // :251
    store_compact(hits, i, hit && best != 0xffffffffu, range_y, best, bu, bv, aux, ray.d.y, ray.d.z);
}

// ---------------------------------------------------------------------------------------------
// Optional ray ordering (TRQ_SORT_RAYS): a counting sort of ray INDICES by (Morton cell of the origin inside the
// scene box, direction octant), so that the rays one warp pulls from the queue start in the same region and head
// the same way. Rays are not moved; hits are still written at the ray's own index; the per-ray traversal is
// untouched, so results are identical with and without it.
#define TRQ_SORT_CELL_BITS 4u                                   // 16^3 cells (B200, C5: 4 bits 829, 5 bits 772, 6 bits 572 Mrays/s)
#define TRQ_SORT_BINS (1u << (3u * TRQ_SORT_CELL_BITS + 3u))    // x 8 octants = 32,768 bins

__device__ __forceinline__ uint32_t spread3(uint32_t v) {       // up to 10 bits -> every third bit
    v &= 0x3ffu;
    v = (v | (v << 16)) & 0x030000ffu;
    v = (v | (v << 8)) & 0x0300f00fu;
    v = (v | (v << 4)) & 0x030c30c3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}

__device__ __forceinline__ uint32_t ray_sort_key(const SceneDev& S, const float4& r0, const float4& r1) {
    const float cells = (float)(1u << TRQ_SORT_CELL_BITS);
    uint32_t c[3];
    const float o[3] = {r0.x, r0.y, r0.z};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float ext = S.rootMax[k] - S.rootMin[k];
        float f = ext > 0.0f ? (o[k] - S.rootMin[k]) / ext * cells : 0.0f;
        f = fminf(fmaxf(f, 0.0f), cells - 1.0f);                // origins outside the scene box clamp to the border cells
        c[k] = (uint32_t)f;
    }
    const uint32_t morton = spread3(c[0]) | (spread3(c[1]) << 1) | (spread3(c[2]) << 2);
    const uint32_t octant = (r1.x < 0.0f ? 1u : 0u) | (r1.y < 0.0f ? 2u : 0u) | (r1.z < 0.0f ? 4u : 0u);
    return (morton << 3) | octant;
}

// Both atomic passes are warp-aggregated (__match_any_sync): lanes with the same key elect one leader that
// issues a single atomicAdd for the group, so a batch whose rays all share one bin (e.g. primary rays from one
// eye point) costs n/32 same-address atomics, not n.
// Automatic mode (no TRQ_SORT_RAYS hint, tree much larger than L2): a probe over 2048 evenly spread runs of 32 consecutive rays
// counts how many neighbouring rays share a key: ctrl[0] = pairs with equal keys, ctrl[2] = pairs looked at. The batch counts as
// INCOHERENT -- worth ordering -- when fewer than half of them do (uniform random rays: ~0; bounce rays off neighbouring pixels:
// ~1/8; primary and shadow rays: nearly all). Every consumer (the three sort passes, the trace kernel) evaluates the same predicate
// from the same two counters, so the decision costs no extra pass and no host round trip; a coherent batch pays the probe and
// three launches that return at once.
__device__ __forceinline__ bool batch_is_incoherent(const uint32_t* ctrl) { return 2u * __ldg(ctrl) < __ldg(ctrl + 2); }

__global__ void __launch_bounds__(256)
sort_probe_kernel(SceneDev S, const trq_ray* __restrict__ rays, uint64_t n, const unsigned long long* __restrict__ nPtr,
                  uint32_t* __restrict__ ctrl) {
    const uint64_t runs = live_count(n, nPtr) / 32u;
    if (runs == 0) return;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5, w = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned lane = threadIdx.x & 31u;
    const uint64_t i = (w * runs / warps) * 32u + lane;
    const float4 r0 = ldg4(reinterpret_cast<const float4*>(rays + i));
    const float4 r1 = ldg4(reinterpret_cast<const float4*>(rays + i) + 1);
    const uint32_t key = ray_sort_key(S, r0, r1);
    const uint32_t next = __shfl_down_sync(0xffffffffu, key, 1);
    const unsigned same = __ballot_sync(0xffffffffu, lane < 31u && next == key);
    if (lane == 0) { atomicAdd(&ctrl[0], (uint32_t)__popc(same)); atomicAdd(&ctrl[2], 31u); }
}

// (count and scatter walk the batch with a grid-stride loop over a capped grid, so that the launches that return at once in
// the automatic mode cost microseconds, not the scheduling of n / 256 empty CTAs)
__global__ void __launch_bounds__(256)
sort_count_kernel(SceneDev S, const trq_ray* __restrict__ rays, uint64_t n, const unsigned long long* __restrict__ nPtr,
                  uint32_t* __restrict__ keys, uint32_t* __restrict__ hist, const uint32_t* __restrict__ ctrl) {
    if (ctrl && !batch_is_incoherent(ctrl)) return;             // automatic mode found the batch coherent: the queue stays as given
    const uint64_t N = live_count(n, nPtr);
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < N; base += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t i = base + threadIdx.x;
        const bool valid = i < N;
        const unsigned vm = __ballot_sync(0xffffffffu, valid);
        if (!valid) continue;
        const float4 r0 = ldg4(reinterpret_cast<const float4*>(rays + i));
        const float4 r1 = ldg4(reinterpret_cast<const float4*>(rays + i) + 1);
        const uint32_t key = ray_sort_key(S, r0, r1);
        keys[i] = key;
        const unsigned peers = __match_any_sync(vm, key);
        if ((threadIdx.x & 31u) == (unsigned)(__ffs(peers) - 1)) atomicAdd(&hist[key], (uint32_t)__popc(peers));
    }
}

// exclusive prefix sum of TRQ_SORT_BINS counters, one CTA of 1024 threads (256 bins per thread)
__global__ void __launch_bounds__(1024)
sort_scan_kernel(uint32_t* __restrict__ hist, const uint32_t* __restrict__ ctrl) {
    __shared__ uint32_t partial[1024];
    if (ctrl && !batch_is_incoherent(ctrl)) return;
    const uint32_t per = TRQ_SORT_BINS / 1024u;
    uint32_t* mine = hist + threadIdx.x * per;
    uint32_t sum = 0;
    for (uint32_t k = 0; k < per; ++k) sum += mine[k];
    partial[threadIdx.x] = sum;
    __syncthreads();
    for (uint32_t off = 1; off < 1024u; off <<= 1) {            // Hillis-Steele inclusive scan
        uint32_t v = threadIdx.x >= off ? partial[threadIdx.x - off] : 0u;
        __syncthreads();
        partial[threadIdx.x] += v;
        __syncthreads();
    }
    uint32_t run = partial[threadIdx.x] - sum;                  // exclusive base of this thread's bins
    for (uint32_t k = 0; k < per; ++k) { const uint32_t c = mine[k]; mine[k] = run; run += c; }
}

__global__ void __launch_bounds__(256)
sort_scatter_kernel(const uint32_t* __restrict__ keys, uint64_t n, const unsigned long long* __restrict__ nPtr,
                    uint32_t* __restrict__ cursor, uint32_t* __restrict__ order, const uint32_t* __restrict__ ctrl) {
    if (ctrl && !batch_is_incoherent(ctrl)) return;
    const uint64_t N = live_count(n, nPtr);
    const unsigned lane = threadIdx.x & 31u;
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < N; base += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t i = base + threadIdx.x;
        const bool valid = i < N;
        const unsigned vm = __ballot_sync(0xffffffffu, valid);
        if (!valid) continue;
        const uint32_t key = keys[i];
        const unsigned peers = __match_any_sync(vm, key);
        const unsigned leader = (unsigned)(__ffs(peers) - 1);
        uint32_t slot = 0;
        if (lane == leader) slot = atomicAdd(&cursor[key], (uint32_t)__popc(peers));
        slot = __shfl_sync(peers, slot, leader);
        order[slot + (uint32_t)__popc(peers & ((1u << lane) - 1u))] = (uint32_t)i;     // lanes keep their index order inside a group
    }
}

// ---------------------------------------------------------------------------------------------
// v1: packed layout, persistent warps, shared-memory far-child stack, records finished in the kernel.

// Output record formats of the packed kernel
enum : int { OUT_HIT32 = 0, OUT_HIT16 = 1 };

struct TraceParams {
    const trq_ray* rays;
    void*          hits;           // trq_hit[n] (OUT_HIT32) or trq_hit16[n] (OUT_HIT16)
    uint64_t       n;
    QueueHead*     queue;          // global ray queue head of this launch (zero on entry, zeroed again by the last CTA)
    uint32_t       stackDepth;     // entries per lane
    uint32_t       refillMin;      // refill when at least this many lanes of a warp are idle
    uint32_t       leafBatch;      // leave the interior phase when this many lanes wait at a leaf
    uint32_t       topCount;       // interior nodes [0, topCount) are staged in shared memory (TOP kernels), else 0
    // 1: launched as a programmatic dependent of the previous kernel on its stream, so its CTAs may start while that
    // kernel's last rays are still being traced. Until a warp has passed griddepcontrol.wait (gate() in the kernel) it
    // stores nothing but into `park`, and it checks every ray it read before the wait again after it.
    uint32_t       early;
    uint32_t       tailSlot;       // TRQ_TAIL_TIMELINE builds: the launch record of g_tail this launch fills
    // trq_profile_enable on an early launch: {start of CTA 0, end of the last CTA} in %globaltimer ns. NULL otherwise.
    unsigned long long* timing;
    // an early launch's scratch for records finished before its wait: [grid warps][TRQ_PARK_ROWS][4][32] float4s, owned by
    // this launch until it ends. NULL: the warps wait after the rays they drew first.
    float4*             park;
    // with park: this launch's word, 0 while it runs (its last CTA sets 1), and the previous launch's on the stream. Warps park
    // only while the previous launch still runs; once it has ended they wait at once (griddepcontrol.wait returns).
    volatile uint32_t*  parkRunning;
    const volatile uint32_t* prevRunning;
    const uint32_t* order;         // optional queue order (TRQ_SORT_RAYS): queue slot -> ray index; NULL = identity
    const uint32_t* orderFlag;     // optional (automatic mode): the probe's counters; `order` applies only if batch_is_incoherent()
    const unsigned long long* nPtr;    // optional device-resident batch size (trq_trace_indirect); n is then the capacity
    // trq_trace_gather: every finished record also counts towards its tile of 2^tileShift consecutive records
    // (tileDone[index >> shift], after a fence), so that the sender kernel -- running beside this kernel -- can ship each
    // tile to the peer GPUs the moment it is complete. NULL otherwise.
    uint32_t*           tileDone;
    uint32_t            tileShift;     // log2(records per tile)
};

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void stg4(void* p, const float4& a) {
    asm volatile("st.global.v4.f32 [%0], {%1,%2,%3,%4};" :: "l"(p), "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w) : "memory");
}
// 256-bit load cached in L2 only. An early launch reads its rays with it: an L1 line filled before griddepcontrol.wait
// may hold what the previous kernel had not yet written, and a later ray of the same line would be read from it.
__device__ __forceinline__ void ldcg8(const float4* p, float4& a, float4& b) {
    asm volatile("ld.global.cg.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "l"(p) : "memory");
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// Programmatic dependent launch (sm_90+). Both are no-ops in a grid that has no programmatic dependency / dependent.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Scratch rows per warp for the records an early launch finishes before its wait (2 KB each). A B200 warp refills about
// every 10-20 us; the previous launch's tail is up to ~200 us (C3, profiles/r07_pdl.txt).
#define TRQ_PARK_ROWS 8u

#ifdef TRQ_TAIL_TIMELINE
// developer instrumentation (tools/build_variant.sh <name> -DTRQ_TAIL_TIMELINE, read by tools/tail_probe.py): per CTA of
// the last TRQ_TAIL_LAUNCHES launches, %globaltimer at {start, ~(first warp to find the queue exhausted), exit}
#define TRQ_TAIL_LAUNCHES 8
#define TRQ_TAIL_MAX_CTAS 4096
__device__ unsigned long long g_tail[TRQ_TAIL_LAUNCHES][TRQ_TAIL_MAX_CTAS][3];
#endif

// trq_hit (two float4) -> trq_hit16 {t, id, u, v}; id = 0xffffffff on a miss, else front << 31 | pType << 28 | pIndex
__device__ __forceinline__ float4 pack_hit16(const float4& o0, const float4& o1) {
    const uint32_t flags = __float_as_uint(o1.w);
    const uint32_t id = (flags & TRQ_HIT_FLAG_HIT)
        ? (((flags & TRQ_HIT_FLAG_FRONT) ? 0x80000000u : 0u) | (__float_as_uint(o0.y) << 28) | (__float_as_uint(o0.z) & 0x0fffffffu))
        : 0xffffffffu;
    return make_float4(o0.x, __uint_as_float(id), o1.x, o1.y);
}

#define TRQ_GATHER_TILE_SHIFT_MIN 8u       // tile sizes a gather may use: 2^8 .. 2^16 records (default 2^11, trq_api.cu)

// One finished record to the output buffer (and, under trq_trace_gather, one more record of its tile complete).
template <int OUT>
__device__ __forceinline__ void emit_record(const TraceParams& P, uint32_t idx, const float4& o0, const float4& o1) {
    if (OUT == OUT_HIT32) stg8(reinterpret_cast<trq_hit*>(P.hits) + idx, o0, o1);
    else                  stg4(reinterpret_cast<float4*>(P.hits) + idx, pack_hit16(o0, o1));
    if (P.tileDone) {
        // the record before the count that announces it; lanes of this warp whose records fall into the same tile (nearly
        // always all of them: a warp draws consecutive queue slots) send ONE count between them -- the whole GPU works on a
        // handful of tiles at any moment, and per-record atomics on those few addresses serialise in L2
        __threadfence();
        const uint32_t tile = idx >> P.tileShift;
        const unsigned peers = __match_any_sync(__activemask(), tile);
        if ((threadIdx.x & 31u) == (unsigned)(__ffs(peers) - 1)) atomicAdd(P.tileDone + tile, (uint32_t)__popc(peers));
    }
}

// Cube::hit_test on the 240-byte reference struct (two per Cornell box: rare). Out of line and fed with scalars by
// value so that the hot loops keep the ray in registers. out = {t, u, v, bits(front | material << 1)}.
// (TAG: one copy per kernel instantiation -- ptxas 12.9 crashes when two entries with different launch bounds share
// an out-of-line function.)
template <int TAG>
__device__ __noinline__ bool leaf_cube(const RefBVH* __restrict__ bvh, const RefCube* __restrict__ cubes, uint32_t leafNode,
                                       float ox, float oy, float oz, float dx, float dy, float dz, float range_y, float4* out) {
    const RayCtx ray = make_ray_ctx(ox, oy, oz, dx, dy, dz);
    float t = 0.0f;
    Surface s;
    if (!cube_hit(&cubes[bvh[leafNode].pIndex], ray, FLT_MIN, range_y, t, &s)) return false;
    *out = make_float4(t, s.uvx, s.uvy, __uint_as_float(s.front | (s.material << 1)));
    return true;
}

// The final trq_hit of a ray that ended on a sphere / square / cube leaf (the triangle case is inline in flush()).
//   sphere: Sphere.hh:51-56 (p, gn = (p - c) / r, checkFace, sphereUV)      square: Square.hh:93-111 (uv, checkFace)
//   cube:   front / material / uv were captured by leaf_cube at hit time
template <int TAG, bool SQCUBE>
__device__ __noinline__ void finish_other(const float4* __restrict__ sph, const float4* __restrict__ sq, const RefBVH* __restrict__ bvh,
                                          uint32_t best, float ox, float oy, float oz, float dx, float dy, float dz,
                                          float t, float u, float v, uint32_t aux, float4* out) {
    const uint32_t kind = TRQ_REF_KIND(best), slot = TRQ_REF_INDEX(best);
    const f3 o = make_f3(ox, oy, oz), d = make_f3(dx, dy, dz);
    float4 o0 = make_float4(0.f, 0.f, 0.f, 0.f), o1 = o0;
    if (kind == REF_SPHERE) {
        float4 s0, s1;
        packed::load_sphere(sph, slot, s0, s1);
        const f3 p = add3(o, scale3(d, t));
        const f3 gn = divs3(sub3(p, make_f3(s0.x, s0.y, s0.z)), s0.w);
        const uint32_t front = front_face(d, gn) ? TRQ_HIT_FLAG_FRONT : 0u;
        const float phi = atan2f(gn.z, gn.x);
        const float theta = asinf(gn.y);
        const float uvx = fsub(1.0f, fdiv(fadd(phi, TRQ_PI_F), fmul(2.0f, TRQ_PI_F)));
        const float uvy = fdiv(fadd(theta, TRQ_PI_2_F), TRQ_PI_F);
        o0 = make_float4(t, __uint_as_float((uint32_t)TRQ_SPHERE), s1.y, s1.x);
        o1 = make_float4(uvx, uvy, s1.z, __uint_as_float(TRQ_HIT_FLAG_HIT | front));
    } else if (SQCUBE && kind == REF_SQUARE) {
        float4 q0, q1, q2;
        packed::load_square(sq, slot, q0, q1, q2);
        const uint32_t axes = __float_as_uint(q1.y);
        const unsigned ai = axes & 3u, aj = (axes >> 8) & 3u, ak = (axes >> 16) & 3u;
        const float a = fadd(get3(o, ai), fmul(t, get3(d, ai)));                   // Square.hh:88,91 with the accepted t
        const float b = fadd(get3(o, aj), fmul(t, get3(d, aj)));
        const float uvx = fdiv(fsub(a, q0.x), fsub(q0.y, q0.x));                   // :96-97
        const float uvy = fdiv(fsub(b, q0.z), fsub(q0.w, q0.z));
        f3 gn = make_f3(0.0f, 0.0f, 0.0f);
        set3(gn, ak, 1.0f);
        const uint32_t front = front_face(d, gn) ? TRQ_HIT_FLAG_FRONT : 0u;       // :99-100
        o0 = make_float4(t, __uint_as_float((uint32_t)TRQ_SQUARE), q2.x, q1.w);
        o1 = make_float4(uvx, uvy, q1.z, __uint_as_float(TRQ_HIT_FLAG_HIT | front));
    } else if (SQCUBE && kind == REF_CUBE) {
        o0 = make_float4(t, __uint_as_float((uint32_t)TRQ_CUBE), __uint_as_float(bvh[slot].pIndex), __uint_as_float(slot));
        o1 = make_float4(u, v, __uint_as_float(aux >> 1), __uint_as_float(TRQ_HIT_FLAG_HIT | ((aux & 1u) ? TRQ_HIT_FLAG_FRONT : 0u)));
    }
    out[0] = o0; out[1] = o1;
}

// Per-ray state that the interior loop never touches is parked in shared memory ([word][BLOCK],
// lane-major => bank-conflict free) so that the hot loop fits in 48 registers (5 resident CTAs of 256 per SM).
enum : uint32_t { COLD_TEST_T = 0, COLD_BEST, COLD_U, COLD_V, COLD_AUX, COLD_RAY, COLD_DX, COLD_DY, COLD_DZ, COLD_WORDS };

#ifndef TRQ_INTERIOR_UNROLL
#define TRQ_INTERIOR_UNROLL 2
#endif
#ifndef TRQ_WAIT_MUL
#define TRQ_WAIT_MUL 2
#endif

#ifdef TRQ_STATS
__device__ unsigned long long g_stats[8];
#endif

// ANY: Scene::hit(any = true). OUT: record format. BLOCK x MINB: CTA size and resident CTAs per SM.
// TOP: the first P.topCount interior nodes are read from shared memory instead of L1/L2.
// LEAVES: which leaf types the tree has. The code of the absent ones is compiled out: a triangle-only kernel has no
//       out-of-line call, no stack frame and no register spill (C3 +4 %, C3 primary +6 %); without Square / Cube leaves the
//       Cube call and its frame go (C1 +5 %, C4 +1 %).
enum : int { LEAVES_ALL = 0, LEAVES_TRI_SPHERE = 1, LEAVES_TRI = 2 };
template <bool ANY, int OUT, int BLOCK, int MINB, bool TOP, int LEAVES>
__global__ void __launch_bounds__(BLOCK, MINB)
trace_packed_kernel(const SceneDev S, const TraceParams P) {
    extern __shared__ __align__(128) uint32_t smem_u32[];
    __shared__ unsigned long long topBarrier;
    const uint32_t topWords = TOP ? packed::staged_words(P.topCount) : 0u;
    const float4* const topNodes = reinterpret_cast<const float4*>(smem_u32);        // [4][topCount]
    uint32_t* const stk = smem_u32 + topWords + threadIdx.x;                         // [stackDepth][BLOCK]
    uint32_t* const cold = smem_u32 + topWords + P.stackDepth * BLOCK + threadIdx.x; // [COLD_WORDS][BLOCK]
    float* const coldf = reinterpret_cast<float*>(cold);
    const unsigned lane = threadIdx.x & 31u;
    constexpr int TAG = ((((BLOCK * 8 + MINB) * 2 + (ANY ? 1 : 0)) * 2 + OUT) * 2 + (TOP ? 1 : 0)) * 4 + LEAVES;
    constexpr bool TRIS = LEAVES == LEAVES_TRI, SQCUBE = LEAVES == LEAVES_ALL;

    // The next trace on this stream may start as this grid's CTAs retire. An early grid lets its own dependent start only
    // once its predecessor has finished (in gate()), so that at most two traces overlap: the queue heads of the ring
    // stay one launch's each.
    bool gated = P.early != 0;                       // this warp has not passed griddepcontrol.wait yet
    bool drew = false;                               // this warp has drawn its first rays
    if (!gated) griddep_launch_dependents();
    if (P.timing && blockIdx.x == 0 && threadIdx.x == 0) P.timing[0] = global_ns();
    if (P.park && blockIdx.x == 0 && threadIdx.x == 0) { *P.parkRunning = 1u; __threadfence(); }
#ifdef TRQ_TAIL_TIMELINE
    unsigned long long* const tail = blockIdx.x < TRQ_TAIL_MAX_CTAS ? g_tail[P.tailSlot % TRQ_TAIL_LAUNCHES][blockIdx.x] : nullptr;
    if (tail && threadIdx.x == 0) tail[0] = global_ns();
#endif
    if (TOP) packed::stage_top_of_tree(reinterpret_cast<float4*>(smem_u32), S.topSoA, P.topCount, S.topStride, &topBarrier);

    const uint64_t N = live_count(P.n, P.nPtr);
    const bool useOrder = P.order != nullptr && (P.orderFlag == nullptr || batch_is_incoherent(P.orderFlag));
    bool active = false, exhausted = false;
    f3 ro = make_f3(0.f, 0.f, 0.f), rinv = make_f3(0.f, 0.f, 0.f);
    float range_y = 0.0f;
    uint32_t cur = TRQ_REF_DONE_WORD, sp = 0;

    // A finished ray only retires its lane; its record is finished and written by flush() when the lane is next given a
    // ray, for all retired lanes at once: the shared-memory reads, the finish-record fetch and the store(s) are then issued
    // once per refill instead of once per finishing ray (most rays finish alone in their warp step). The lane's
    // registers (ro, range_y) stay untouched between finish() and flush().
    bool pending = false;
    auto finish = [&]() { active = false; pending = true; };
    auto record = [&](float4& o0, float4& o1) {                       // the finished ray's record
            const uint32_t best = cold[COLD_BEST * BLOCK];
            const bool hit = (range_y < coldf[COLD_TEST_T * BLOCK]) && best != 0xffffffffu;   // Render.hh:251
            o0 = make_float4(0.f, 0.f, 0.f, 0.f); o1 = o0;
            if (hit) {
                const float u = coldf[COLD_U * BLOCK], v = coldf[COLD_V * BLOCK];
                const f3 d = make_f3(coldf[COLD_DX * BLOCK], coldf[COLD_DY * BLOCK], coldf[COLD_DZ * BLOCK]);
                if (TRQ_REF_KIND(best) == REF_TRI) {
                    // Triangle.hh:73-82: interpolated normal, checkFace; ids from the finish record
                    float4 q0, q1, q2;
                    packed::load_tri_finish(S.triN, TRQ_REF_INDEX(best), q0, q1, q2);
                    const float w = fsub(fsub(1.0f, u), v);
                    const f3 gn = add3(add3(scale3(make_f3(q1.x, q1.y, q1.z), u), scale3(make_f3(q2.x, q2.y, q2.z), v)),
                                       scale3(make_f3(q0.x, q0.y, q0.z), w));
                    const uint32_t front = front_face(d, gn) ? TRQ_HIT_FLAG_FRONT : 0u;
                    o0 = make_float4(range_y, __uint_as_float((uint32_t)TRQ_TRIANGLE), q1.w, q0.w);
                    o1 = make_float4(u, v, __uint_as_float(19u), __uint_as_float(TRQ_HIT_FLAG_HIT | front));
                } else if (!TRIS) {
                    float4 o[2];
                    finish_other<TAG, SQCUBE>(S.sph, S.sq, S.bvh, best, ro.x, ro.y, ro.z, d.x, d.y, d.z, range_y, u, v, cold[COLD_AUX * BLOCK], o);
                    o0 = o[0]; o1 = o[1];
                }
            }
    };
    auto flush = [&]() {
        if (pending) {
            float4 o0, o1;
            record(o0, o1);
            emit_record<OUT>(P, cold[COLD_RAY * BLOCK], o0, o1);
            pending = false;
        }
    };
    // Before its wait an early warp may store nothing where the caller can see it: the previous kernel may still read or
    // write those buffers. It parks the records of its finished rays instead, one row of 32 per refill, in this launch's own
    // scratch (P.park): [warp][row][quarter][lane] float4s = {ox, oy, oz, tmax}, {dx, dy, dz, bits(ray index)}, the record's
    // two halves; ray index ~0: no ray. After the wait, gate() stores each parked record whose ray is still what was traced.
    const uint64_t parkWarp = ((uint64_t)blockIdx.x * (BLOCK / 32) + (threadIdx.x >> 5)) * TRQ_PARK_ROWS;
    uint32_t parked = 0;                             // rows this warp has parked
    uint32_t redo = 0;                               // this lane's parked rows whose ray changed: traced again after the wait
    auto park = [&]() {
        float4* const row = P.park + (parkWarp + parked) * 128u + lane;
        float4 q1 = make_float4(0.f, 0.f, 0.f, __uint_as_float(0xffffffffu));
        if (pending) {
            float4 o0, o1;
            record(o0, o1);
            stg4(row, make_float4(ro.x, ro.y, ro.z, coldf[COLD_TEST_T * BLOCK]));
            q1 = make_float4(coldf[COLD_DX * BLOCK], coldf[COLD_DY * BLOCK], coldf[COLD_DZ * BLOCK], __uint_as_float(cold[COLD_RAY * BLOCK]));
            stg4(row + 64, o0);
            stg4(row + 96, o1);
            pending = false;
        }
        stg4(row + 32, q1);
        ++parked;
    };
    auto push = [&](uint32_t ref) { stk[sp * BLOCK] = ref; ++sp; };
    auto pop = [&]() {
        if (sp == 0) cur = TRQ_REF_DONE_WORD; else { --sp; cur = stk[sp * BLOCK]; }
    };
    // Draws `want` queue slots for the lanes in `mask` (one atomic per warp) and returns this lane's ray index, or ~0.
    auto draw = [&](unsigned mask) -> uint64_t {
        const int want = __popc(mask);
#ifdef TRQ_STATS
        if (lane == 0) { atomicAdd(&g_stats[4], 1ull); atomicAdd(&g_stats[5], (unsigned long long)want); }
#endif
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(&P.queue->head, (unsigned long long)want);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base + (unsigned long long)want >= N) {
#ifdef TRQ_TAIL_TIMELINE
            if (tail && lane == 0 && !exhausted) atomicMax(&tail[1], ~global_ns());     // stored inverted: 0 = never
#endif
            exhausted = true;
        }
        const uint64_t slot = base + (uint64_t)__popc(mask & ((1u << lane) - 1u));
        if (!((mask >> lane) & 1u) || slot >= N) return ~0ull;
        return useOrder ? (uint64_t)__ldg(P.order + slot) : slot;
    };
    // Gives this lane ray `idx` (r0, r1: its trq_ray). A ray that misses the root is finished at once: its (all-zero)
    // record is stored now, or -- `defer`, in an early launch -- left pending for flush(), like any finished ray.
    auto start = [&](uint32_t idx, const float4& r0, const float4& r1, bool defer) {
        const RayCtx ray = make_ray_ctx(r0.x, r0.y, r0.z, r1.x, r1.y, r1.z);
        ro = ray.o; rinv = ray.inv;
        range_y = r0.w;                                                // Render.hh:143  range_t = (FLT_MIN, test_t)
        sp = 0;
        const f3 rootMin = make_f3(S.rootMin[0], S.rootMin[1], S.rootMin[2]);
        const f3 rootMax = make_f3(S.rootMax[0], S.rootMax[1], S.rootMax[2]);
        const bool root = box_hit(rootMin, rootMax, ray, FLT_MIN, range_y);    // :145
        if (root || defer) {
            coldf[COLD_TEST_T * BLOCK] = r0.w;
            cold[COLD_BEST * BLOCK] = 0xffffffffu;
            coldf[COLD_U * BLOCK] = 0.0f; coldf[COLD_V * BLOCK] = 0.0f;
            cold[COLD_AUX * BLOCK] = 0u;
            cold[COLD_RAY * BLOCK] = idx;
            coldf[COLD_DX * BLOCK] = r1.x; coldf[COLD_DY * BLOCK] = r1.y; coldf[COLD_DZ * BLOCK] = r1.z;
        }
        if (root) { cur = S.rootRef; active = true; }
        else if (defer) pending = true;
        else {
            const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
            emit_record<OUT>(P, idx, z, z);
        }
    };
    // An early warp's wait for the previous kernel on the stream (it returns once that grid has finished and its stores
    // are visible). The rays this warp drew before it may have been read before the previous kernel wrote them (a caller's
    // kernel that rewrites the batch, or a batch that is the previous trace's output): every lane reads its ray again and
    // starts it over if any of the seven words the traversal uses (flags is reserved) has changed.
    auto gate = [&]() {
        griddep_wait();
        griddep_launch_dependents();
        gated = false;
        for (uint32_t r = 0; r < parked; ++r) {
            const float4* const row = P.park + (parkWarp + r) * 128u + lane;
            const float4 q1 = __ldcg(row + 32);
            const uint32_t idx = __float_as_uint(q1.w);
            if (idx == 0xffffffffu) continue;
            const float4 q0 = __ldcg(row);
            float4 r0, r1;
            ldcg8(reinterpret_cast<const float4*>(P.rays + idx), r0, r1);
            const bool same = __float_as_uint(r0.x) == __float_as_uint(q0.x) && __float_as_uint(r0.y) == __float_as_uint(q0.y) &&
                              __float_as_uint(r0.z) == __float_as_uint(q0.z) && __float_as_uint(r0.w) == __float_as_uint(q0.w) &&
                              __float_as_uint(r1.x) == __float_as_uint(q1.x) && __float_as_uint(r1.y) == __float_as_uint(q1.y) &&
                              __float_as_uint(r1.z) == __float_as_uint(q1.z);
            if (same) emit_record<OUT>(P, idx, __ldcg(row + 64), __ldcg(row + 96));
            else      redo |= 1u << r;
        }
        if (active || pending) {
            const uint32_t idx = cold[COLD_RAY * BLOCK];
            float4 r0, r1;
            ldcg8(reinterpret_cast<const float4*>(P.rays + idx), r0, r1);
            const bool same = __float_as_uint(r0.x) == __float_as_uint(ro.x) && __float_as_uint(r0.y) == __float_as_uint(ro.y) &&
                              __float_as_uint(r0.z) == __float_as_uint(ro.z) && __float_as_uint(r0.w) == cold[COLD_TEST_T * BLOCK] &&
                              __float_as_uint(r1.x) == cold[COLD_DX * BLOCK] && __float_as_uint(r1.y) == cold[COLD_DY * BLOCK] &&
                              __float_as_uint(r1.z) == cold[COLD_DZ * BLOCK];
            if (!same) { active = false; pending = false; start(idx, r0, r1, true); }
        }
    };

    for (;;) {
        // ---- refill idle lanes from the global queue: one atomic per warp ----
        unsigned idleMask = __ballot_sync(0xffffffffu, !active);
        bool more = !exhausted || __any_sync(0xffffffffu, redo != 0u);
        bool refill = more && (idleMask == 0xffffffffu || __popc(idleMask) >= (int)P.refillMin);
        // an early warp parks its finished rays' records while it has scratch rows left, then waits
        if (refill && gated && drew &&
            (P.park == nullptr || parked == TRQ_PARK_ROWS || __shfl_sync(0xffffffffu, lane == 0 ? *P.prevRunning : 0u, 0) == 0u)) {
            gate();
            idleMask = __ballot_sync(0xffffffffu, !active);
            more = !exhausted || __any_sync(0xffffffffu, redo != 0u);
            refill = more && (idleMask == 0xffffffffu || __popc(idleMask) >= (int)P.refillMin);
        }
        if (refill) {
            drew = true;
            const bool again = !active && redo != 0u;          // an idle lane with a parked ray that changed traces it first
            const unsigned drawMask = idleMask & ~__ballot_sync(0xffffffffu, again);
            uint64_t idx = ~0ull;
            if (drawMask != 0u && !exhausted) idx = draw(drawMask);
            if (gated) { if (__any_sync(0xffffffffu, pending)) park(); }
            else flush();
            if (again) {
                const uint32_t r = (uint32_t)__ffs(redo) - 1u;
                redo &= redo - 1u;
                idx = __float_as_uint(__ldcg(P.park + (parkWarp + r) * 128u + 32u + lane).w);
            }
            if (idx != ~0ull) {
                float4 r0, r1;                                         // trq_ray is one 32-byte record
                if (P.early) ldcg8(reinterpret_cast<const float4*>(P.rays + idx), r0, r1);
                else         ldg8(reinterpret_cast<const float4*>(P.rays + idx), r0, r1);
                start((uint32_t)idx, r0, r1, gated);
            }
        }
        const unsigned actMask = __ballot_sync(0xffffffffu, active);
        if (actMask == 0u) {
            if (!exhausted) continue;
            if (gated) gate();
            if (__any_sync(0xffffffffu, active || redo != 0u)) continue;   // rays that changed start over
            flush();
            break;
        }

        // ---- traverse until enough lanes have retired to make a refill worthwhile ----
        // Two phases per round so that the (rarer) leaf code is not issued on every interior step:
        //   interior phase: lanes sitting on an interior node step; lanes that reached a leaf wait (a lane
        //     must test its leaf BEFORE it continues, or pruning/tie order would differ from the reference);
        //     the phase ends when no lane is on an interior node or enough lanes wait at leaves;
        //   leaf phase: every waiting lane tests its primitive and pops.
        const int keepGoing = exhausted ? 0 : (32 - (int)P.refillMin);
        do {
            for (;;) {
                const bool onInterior = active && TRQ_REF_KIND(cur) == REF_INTERIOR;
                const int nInt = __popc(__ballot_sync(0xffffffffu, onInterior));
                const int nWait = __popc(__ballot_sync(0xffffffffu, active && !onInterior));
                // leave the interior phase once the lanes waiting at a leaf are more than half of those still stepping
                // (B200 sweep, C3 / 1 M soup Mrays/s: never 4094 / 1141, nWait > nInt 4650 / 1154, 2 nWait > nInt 4727 / 1158,
                // 3x 4701 / 1157, 4x 4678 / 1158, 6x 4614 / 1155)
                if (nInt == 0 || nWait >= (int)P.leafBatch || TRQ_WAIT_MUL * nWait > nInt) break;
#pragma unroll
                for (int rep = 0; rep < TRQ_INTERIOR_UNROLL; ++rep) {          // steps per vote round
#ifdef TRQ_STATS
                    { const unsigned m_ = __ballot_sync(0xffffffffu, active && TRQ_REF_KIND(cur) == REF_INTERIOR);
                      if (lane == 0 && m_) { atomicAdd(&g_stats[0], 1ull); atomicAdd(&g_stats[1], (unsigned long long)__popc(m_)); }
                      const unsigned t_ = __ballot_sync(0xffffffffu, active && TRQ_REF_KIND(cur) == REF_INTERIOR && TOP && TRQ_REF_INDEX(cur) < P.topCount);
                      if (lane == 0 && t_) atomicAdd(&g_stats[6], (unsigned long long)__popc(t_)); }
#endif
                    if (active && TRQ_REF_KIND(cur) == REF_INTERIOR) {
                        const uint32_t ni = TRQ_REF_INDEX(cur);
                        float4 q0, q1, q2, q3;
                        if (TOP && ni < P.topCount) packed::load_staged_node(topNodes, P.topCount, ni, q0, q1, q2, q3);   // this CTA's copy
                        else                        packed::load_node(S.nodes, ni, q0, q1, q2, q3);
                        float tl = range_y, tr = range_y;                     // :157
                        const bool lt = box_entry(make_f3(q0.x, q0.y, q0.z), make_f3(q1.x, q1.y, q1.z), ro, rinv, range_y, tl);   // :159
                        const bool rt = box_entry(make_f3(q2.x, q2.y, q2.z), make_f3(q3.x, q3.y, q3.z), ro, rinv, range_y, tr);   // :160
                        const uint32_t lref = __float_as_uint(q0.w), rref = __float_as_uint(q1.w);
                        if (!lt && !rt) {                                     // :162-169  pop
                            pop();
                        } else {
                            const bool selLeft = tl < tr;                     // :174 (ties -> right, quirk included)
                            if (lt && rt) push(selLeft ? rref : lref);        // :171-172
                            cur = selLeft ? lref : rref;
                        }
                        if (cur == TRQ_REF_DONE_WORD) finish();
                    }
                }
            }
#ifdef TRQ_STATS
            { const unsigned m_ = __ballot_sync(0xffffffffu, active && TRQ_REF_KIND(cur) != REF_INTERIOR);
              if (lane == 0 && m_) { atomicAdd(&g_stats[2], 1ull); atomicAdd(&g_stats[3], (unsigned long long)__popc(m_)); } }
#endif
            if (active && TRQ_REF_KIND(cur) != REF_INTERIOR) {
                const uint32_t kind = TRQ_REF_KIND(cur);
                RayCtx ray;
                ray.o = ro; ray.inv = rinv;
                ray.d = make_f3(coldf[COLD_DX * BLOCK], coldf[COLD_DY * BLOCK], coldf[COLD_DZ * BLOCK]);
                bool h = false; float t = 0.0f, u = 0.0f, v = 0.0f; uint32_t a = 0;
                if (kind == REF_TRI) {
                    float4 t0, t1, t2;
                    packed::load_tri(S.tris, TRQ_REF_INDEX(cur), t0, t1, t2);
                    h = tri_hit(make_f3(t0.x, t0.y, t0.z), make_f3(t1.x, t1.y, t1.z), make_f3(t2.x, t2.y, t2.z),
                                ray, FLT_MIN, range_y, t, u, v);
                }
                else if (!TRIS && kind == REF_SPHERE) {
                    const float4 s0 = packed::load_sphere_test(S.sph, TRQ_REF_INDEX(cur));
                    h = sphere_hit(make_f3(s0.x, s0.y, s0.z), s0.w, ray, FLT_MIN, range_y, t);
                } else if (SQCUBE && kind == REF_SQUARE) {
                    // Square::hit_test (Square.hh:82-92) on the packed record; the rejections are pure comparisons, and-ed
                    float4 q0, q1;
                    packed::load_square_test(S.sq, TRQ_REF_INDEX(cur), q0, q1);
                    const uint32_t axes = __float_as_uint(q1.y);
                    const unsigned ai = axes & 3u, aj = (axes >> 8) & 3u, ak = (axes >> 16) & 3u;
                    const float tt = fdiv(fsub(q1.x, get3(ro, ak)), get3(ray.d, ak));
                    bool ok = !(isinf(tt) || isnan(tt)) && !(tt < FLT_MIN || tt > range_y);
                    const float sa = fadd(get3(ro, ai), fmul(tt, get3(ray.d, ai)));
                    ok = ok && !(sa < q0.x || sa > q0.y);
                    const float sb = fadd(get3(ro, aj), fmul(tt, get3(ray.d, aj)));
                    ok = ok && !(sb < q0.z || sb > q0.w);
                    if (ok) { h = true; t = tt; }
                } else if (SQCUBE && kind == REF_CUBE) {
                    float4 o4;
                    h = leaf_cube<TAG>(S.bvh, S.cubes, TRQ_REF_INDEX(cur), ro.x, ro.y, ro.z, ray.d.x, ray.d.y, ray.d.z, range_y, &o4);
                    if (h) { t = o4.x; u = o4.y; v = o4.z; a = __float_as_uint(o4.w); }
                }
                if (h) {
                    range_y = t;
                    cold[COLD_BEST * BLOCK] = cur;
                    coldf[COLD_U * BLOCK] = u; coldf[COLD_V * BLOCK] = v;
                    cold[COLD_AUX * BLOCK] = a;
                }
                if (ANY && range_y < coldf[COLD_TEST_T * BLOCK]) cur = TRQ_REF_DONE_WORD;   // :244
                else pop();
                if (cur == TRQ_REF_DONE_WORD) finish();
            }
        } while (__popc(__ballot_sync(0xffffffffu, active)) > keepGoing);
    }

    // ---- epilogue (every warp has passed gate()): the last CTA to leave re-arms the queue head for the next launch that draws it
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int prev = atomicAdd(&P.queue->done, 1u);
        if (prev == gridDim.x - 1) {
            if (P.timing) P.timing[1] = global_ns();
            if (P.park) *P.parkRunning = 0u;
            P.queue->head = 0ull;
            P.queue->done = 0u;
        }
#ifdef TRQ_TAIL_TIMELINE
        if (tail) tail[2] = global_ns();
#endif
    }
}

// ---------------------------------------------------------------------------------------------
// trq_trace_gather, the collective half. Runs BESIDE trace_packed_kernel on a second stream (one 128-thread, 32-register
// CTA per SM fits next to the five resident trace CTAs) and ships this rank's records to every peer GPU tile by tile, as
// soon as the trace has finished a tile: coalesced 16-byte loads from the local buffer (L2), coalesced 16-byte stores into
// the same place of every peer's buffer over NVLink. The all-gather therefore runs under the traversal instead of after it,
// and with full-line stores instead of one 32-byte store per ray (per-ray peer stores from the trace kernel itself reached
// 371 GB/s of NVLink egress at 8 GPUs; coalesced tiles reach the 650-700 GB/s the resolve-pass gather of round 1 did).
// The last CTA to finish publishes (count, step) to every rank with system-scope release stores.
struct SendParams {
    const uint4*        src;                               // this rank's slot of its own buffer (records as 16-byte units)
    uint4*              peer[TRQ_MAX_PEERS];               // the same slot in every other rank's buffer
    unsigned long long* peerFlag[TRQ_MAX_PEERS];           // flags[rank] on every other rank: last completed step
    unsigned long long* peerCount[TRQ_MAX_PEERS];          // counts[phase][rank] on every other rank
    unsigned long long* ownFlag;
    unsigned long long* ownCount;
    const uint32_t*     tileDone;                          // records finished per tile (written by the trace kernel)
    unsigned int*       blocksDone;
    unsigned int*       status;                            // raised (mapped host memory) if the trace never delivers a tile
    unsigned long long  n, step, timeoutNs;
    uint32_t            nPeer, unitsPerRecord;             // 2 for trq_hit, 1 for trq_hit16
    uint32_t            tileShift;
};

__device__ __forceinline__ uint32_t ld_acquire_gpu_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(128, 16)
gather_send_kernel(const SendParams G) {
    // (no shared memory: the CTA has to fit into what five resident trace CTAs leave of the SM's carve-out)
    const uint64_t tileRecords = 1ull << G.tileShift;
    const uint64_t nTiles = (G.n + tileRecords - 1) >> G.tileShift;
    for (uint64_t tile = blockIdx.x; tile < nTiles; tile += gridDim.x) {
        const uint64_t first = tile << G.tileShift;
        const uint32_t count = (uint32_t)((G.n - first) < tileRecords ? (G.n - first) : tileRecords);
        int giveUp = 0;
        if (threadIdx.x == 0) {                              // wait until the trace has finished every record of this tile
            unsigned long long t0;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
            while (ld_acquire_gpu_u32(G.tileDone + tile) < count) {
                unsigned long long t;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
                if (t - t0 > G.timeoutNs) { *G.status = 0x80000000u; giveUp = 1; break; }
                __nanosleep(200);
            }
        }
        if (__syncthreads_or(giveUp)) break;
        const uint64_t base = first * G.unitsPerRecord, total = (uint64_t)count * G.unitsPerRecord;
        for (uint64_t i = threadIdx.x; i < total; i += 256) {     // two 16-byte units in flight per thread
            const uint4 a = __ldcg(G.src + base + i);
            const bool two = i + 128 < total;
            const uint4 b = two ? __ldcg(G.src + base + i + 128) : a;
#pragma unroll 1
            for (uint32_t p = 0; p < G.nPeer; ++p) {
                G.peer[p][base + i] = a;
                if (two) G.peer[p][base + i + 128] = b;
            }
        }
    }
    __threadfence_system();                                   // this thread's peer stores before the CTA's arrival
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int prev = atomicAdd(G.blocksDone, 1u);
        if (prev == gridDim.x - 1) {                          // last CTA: every record of this rank is on its way
            *G.blocksDone = 0u;
            __threadfence_system();
            *G.ownCount = G.n;
            st_release_sys(G.ownFlag, G.step);
#pragma unroll 1
            for (uint32_t p = 0; p < G.nPeer; ++p) {
                *G.peerCount[p] = G.n;
                st_release_sys(G.peerFlag[p], G.step);
            }
        }
    }
}

// The same sender with the copy engine of the SM doing the work (the default; TRQ_GATHER_TMA=0 selects the one above): one thread per CTA drives TMA bulk copies
// (cp.async.bulk): tile chunk -> shared memory (completion on an mbarrier), shared memory -> the slot in every peer's
// buffer over NVLink (bulk async-groups), two chunks in flight. No registers or LSU slots per byte in flight -- the l1tex
// pipe the trace kernel is bound by is left alone -- and the NVLink writes are full 128-byte lines issued in long bursts.
#define TRQ_SEND_TMA_STAGES 2u
#define TRQ_SEND_TMA_CHUNK 12288u          // bytes per stage (2 x 12 KB + 1 KB reserve fit beside the trace CTAs' carve-out)

__global__ void __launch_bounds__(32)
gather_send_tma_kernel(const SendParams G) {
    extern __shared__ __align__(128) unsigned char sendBuf[];           // [TRQ_SEND_TMA_STAGES][TRQ_SEND_TMA_CHUNK]
    __shared__ __align__(8) unsigned long long loadBar[TRQ_SEND_TMA_STAGES];
    if (threadIdx.x == 0) {
        for (uint32_t k = 0; k < TRQ_SEND_TMA_STAGES; ++k)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"((uint32_t)__cvta_generic_to_shared(&loadBar[k])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const uint64_t tileRecords = 1ull << G.tileShift;
        const uint64_t nTiles = (G.n + tileRecords - 1) >> G.tileShift;
        const uint32_t recBytes = G.unitsPerRecord * 16u;
        uint32_t chunkNo = 0;                                             // chunks issued so far: stage = chunkNo % stages
        bool giveUp = false;
        for (uint64_t tile = blockIdx.x; tile < nTiles && !giveUp; tile += gridDim.x) {
            const uint64_t first = tile << G.tileShift;
            const uint32_t count = (uint32_t)((G.n - first) < tileRecords ? (G.n - first) : tileRecords);
            unsigned long long t0;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
            while (ld_acquire_gpu_u32(G.tileDone + tile) < count) {      // the trace has finished every record of this tile
                unsigned long long t;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
                if (t - t0 > G.timeoutNs) { *G.status = 0x80000000u; giveUp = true; break; }
                __nanosleep(200);
            }
            if (giveUp) break;
            // records written by st.global on other SMs, read here by the async proxy: order the two
            asm volatile("fence.proxy.async.global;" ::: "memory");
            const uint64_t tileBytes = (uint64_t)count * recBytes, base = first * recBytes;
            for (uint64_t off = 0; off < tileBytes; off += TRQ_SEND_TMA_CHUNK, ++chunkNo) {
                const uint32_t bytes = (uint32_t)((tileBytes - off) < TRQ_SEND_TMA_CHUNK ? (tileBytes - off) : TRQ_SEND_TMA_CHUNK);
                const uint32_t stage = chunkNo % TRQ_SEND_TMA_STAGES, phase = (chunkNo / TRQ_SEND_TMA_STAGES) & 1u;
                const uint32_t sm = (uint32_t)__cvta_generic_to_shared(sendBuf + stage * TRQ_SEND_TMA_CHUNK);
                const uint32_t mb = (uint32_t)__cvta_generic_to_shared(&loadBar[stage]);
                // the peer stores that last read this stage must have read it
                asm volatile("cp.async.bulk.wait_group.read %0;" :: "n"(TRQ_SEND_TMA_STAGES - 1) : "memory");
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mb), "r"(bytes) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             :: "r"(sm), "l"(reinterpret_cast<const unsigned char*>(G.src) + base + off), "r"(bytes), "r"(mb) : "memory");
                uint32_t ready = 0;
                while (!ready)
                    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                                 : "=r"(ready) : "r"(mb), "r"(phase) : "memory");
#pragma unroll 1
                for (uint32_t p = 0; p < G.nPeer; ++p)
                    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                 :: "l"(reinterpret_cast<unsigned char*>(G.peer[p]) + base + off), "r"(sm), "r"(bytes) : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        }
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");       // every peer store of this CTA has been performed
        asm volatile("fence.proxy.async.global;" ::: "memory");
        __threadfence_system();
        const unsigned int prev = atomicAdd(G.blocksDone, 1u);
        if (prev == gridDim.x - 1) {                          // last CTA: every record of this rank is on its way
            *G.blocksDone = 0u;
            __threadfence_system();
            *G.ownCount = G.n;
            st_release_sys(G.ownFlag, G.step);
#pragma unroll 1
            for (uint32_t p = 0; p < G.nPeer; ++p) {
                *G.peerCount[p] = G.n;
                st_release_sys(G.peerFlag[p], G.step);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// compact -> trq_hit, in place, for the reference-layout kernel (the packed kernel finishes its own records).
// One thread per ray, fully coalesced.
__global__ void __launch_bounds__(256)
resolve_hits_kernel(SceneDev S, const trq_ray* __restrict__ rays, trq_hit* hits, uint64_t n, const unsigned long long* __restrict__ nPtr) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= live_count(n, nPtr)) return;
    float4* io = reinterpret_cast<float4*>(hits + i);
    const float4 a = io[0], b = io[1];
    trq_hit out;
    out.t = 0.0f; out.pType = 0; out.pIndex = 0; out.leafNode = 0; out.u = 0.0f; out.v = 0.0f; out.material = 0; out.flags = 0;
    if (__float_as_uint(b.y) != 0u) {
        const uint32_t leaf = __float_as_uint(a.y);
        const int32_t pType = S.bvh[leaf].pType;
        const uint32_t pIndex = S.bvh[leaf].pIndex;
        RayCtx ray;
        if (pType == TRQ_TRIANGLE) {                          // only the direction matters (checkFace), and the trace kernel left it here
            ray = make_ray_ctx(0.0f, 0.0f, 0.0f, b.x, b.z, b.w);
        } else {
            const float4 r0 = ldg4(reinterpret_cast<const float4*>(rays + i));
            const float4 r1 = ldg4(reinterpret_cast<const float4*>(rays + i) + 1);
            ray = make_ray_ctx(r0.x, r0.y, r0.z, r1.x, r1.y, r1.z);
        }
        out.t = a.x; out.pType = (uint32_t)pType; out.pIndex = pIndex; out.leafNode = leaf;
        Surface s; s.front = 0; s.material = 0; s.uvx = s.uvy = 0.0f;
        if (pType == TRQ_TRIANGLE) {
            tri_surface(S.verts, S.idx, pIndex, a.z, a.w, ray, s);
            out.u = a.z; out.v = a.w;
        } else if (pType == TRQ_SPHERE) {
            sphere_surface(&S.spheres[pIndex], a.x, ray, s);
            out.u = s.uvx; out.v = s.uvy;
        } else if (pType == TRQ_SQUARE) {
            float t;
            square_hit(&S.squares[pIndex], ray, a.x, a.x, t, &s);          // same t -> same a, b, uv
            out.u = s.uvx; out.v = s.uvy;
        } else if (pType == TRQ_CUBE) {
            const uint32_t aux = __float_as_uint(b.x);
            s.front = aux & 1u; s.material = aux >> 1;
            out.u = a.z; out.v = a.w;
        }
        out.material = s.material;
        out.flags = TRQ_HIT_FLAG_HIT | (s.front ? TRQ_HIT_FLAG_FRONT : 0u);
    }
    float4 o0, o1;
    o0.x = out.t; o0.y = __uint_as_float(out.pType); o0.z = __uint_as_float(out.pIndex); o0.w = __uint_as_float(out.leafNode);
    o1.x = out.u; o1.y = out.v; o1.z = __uint_as_float(out.material); o1.w = __uint_as_float(out.flags);
    io[0] = o0; io[1] = o1;
}

// Waits (on the stream) until every rank has published `step`; gives up after timeoutNs and raises *status.
__global__ void gather_wait_kernel(const unsigned long long* flags, uint32_t world, unsigned long long step,
                                   unsigned long long timeoutNs, volatile unsigned int* status) {
    const uint32_t p = threadIdx.x;
    if (p >= world) return;
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (ld_acquire_sys(flags + p) < step) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if (t - t0 > timeoutNs) { *status = 1u + p; break; }
        __nanosleep(256);
    }
}

// trq_hit -> HitRecord fields.
__global__ void __launch_bounds__(256)
expand_hits_kernel(SceneDev S, const trq_ray* __restrict__ rays, const trq_hit* __restrict__ hits,
                   trq_hit_record* __restrict__ recs, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const trq_hit h = hits[i];
    trq_hit_record out;
    out.hit = 0; out.t = 0.0f; out.front = 0; out.material = 0; out.pad = 0;
    out.p[0] = out.p[1] = out.p[2] = 0.0f; out.gn[0] = out.gn[1] = out.gn[2] = 0.0f;
    out.sn[0] = out.sn[1] = out.sn[2] = 0.0f; out.uv[0] = out.uv[1] = 0.0f;
    if (h.flags & TRQ_HIT_FLAG_HIT) {
        const float4 r0 = ldg4(reinterpret_cast<const float4*>(rays + i));
        const float4 r1 = ldg4(reinterpret_cast<const float4*>(rays + i) + 1);
        const RayCtx ray = make_ray_ctx(r0.x, r0.y, r0.z, r1.x, r1.y, r1.z);
        Surface s; s.p = s.gn = s.sn = make_f3(0.f, 0.f, 0.f); s.uvx = s.uvy = 0.0f; s.front = 0; s.material = 0;
        float t;
        if (h.pType == TRQ_TRIANGLE)     tri_surface(S.verts, S.idx, h.pIndex, h.u, h.v, ray, s);
        else if (h.pType == TRQ_SPHERE)  sphere_surface(&S.spheres[h.pIndex], h.t, ray, s);
        else if (h.pType == TRQ_SQUARE)  square_hit(&S.squares[h.pIndex], ray, h.t, h.t, t, &s);
        else if (h.pType == TRQ_CUBE)    cube_surface(&S.cubes[h.pIndex], ray, h.t, h.u, h.v, s);
        out.hit = 1; out.t = h.t;
        out.p[0] = s.p.x; out.p[1] = s.p.y; out.p[2] = s.p.z;
        out.gn[0] = s.gn.x; out.gn[1] = s.gn.y; out.gn[2] = s.gn.z;
        out.sn[0] = s.sn.x; out.sn[1] = s.sn.y; out.sn[2] = s.sn.z;
        out.uv[0] = s.uvx; out.uv[1] = s.uvy;
        out.front = s.front; out.material = s.material;
    }
    recs[i] = out;
}

}  // namespace trq
