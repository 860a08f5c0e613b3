/* include/tracer_rq.h -- C-ABI of the B200-native ray-query engine ("trq").
 *
 * Drop-in boundary for the ONE hot path of iaomw/Tracer this repository replaces: the
 * RT_Metal ray query. Everything crossing this boundary is a plain pointer + size in the
 * reference's own byte layouts; there are no torch / C++ types in any signature.
 *
 *   reference interface                                      replaced by
 *   -------------------------------------------------------  ---------------------------
 *   struct Primitive (6 device pointers)                     trq_scene_desc
 *       RT_Metal/Metal/Render.hh:122-130
 *   newBufferWithBytes idx / tri / bvh  (host->device seam)  trq_scene_create
 *       RT_Metal/Tracer/AAPLRenderer.mm:217-231,614-624
 *   argumentEncoderPri setBuffer x6                          (held inside trq_scene)
 *       RT_Metal/Tracer/AAPLRenderer.mm:712-720
 *   bool Scene::hit(ray, hitRecord, test_t, any)             trq_trace (one call = a batch of rays)
 *       RT_Metal/Metal/Render.hh:132-252
 *   struct Ray   RT_Metal/Metal/Ray.hh:10-33                 trq_ray  (first 32 B of Ray; tmax = test_t)
 *   struct HitRecord  RT_Metal/Metal/HitRecord.hh:9-30       trq_hit (compact, + primitive id) and
 *                                                            trq_hit_record via trq_expand_hits
 *   BVH::buildNode / BVH::buildTree (host)                   trq_bvh_build_node(s) / trq_bvh_build_tree
 *       RT_Metal/Metal/BVH.hh:246-314
 *
 * Scene arrays use the reference byte layouts (Metal / Apple-simd rules, float3 = 16 B):
 *   BVH 64 B (BVH.hh:15-22), AABB 32 B (AABB.hh:7-9), TriangleVertex 32 B (Triangle.hh:12-18),
 *   Sphere 272 B (Sphere.hh:6-15), Square 272 B (Square.hh:12-27), Cube 240 B (Cube.hh:6-13).
 *
 * Results are bit-identical to the reference's Scene::hit evaluated in strict IEEE fp32
 * (hit flag, t, primitive id, barycentrics): same per-ray visit order, same arithmetic.
 *
 * Error convention: every call returns TRQ_OK (0) or a negative trq_status; no C++
 * exception crosses the ABI; trq_last_error_string() describes the last failure on the
 * calling thread. There is no CPU fallback: without a CUDA device every compute entry
 * point fails with TRQ_ERR_NO_DEVICE.
 */
#ifndef TRACER_RQ_H
#define TRACER_RQ_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRQ_VERSION 200  /* 0.2.0 */

typedef enum trq_status {
    TRQ_OK            =  0,
    TRQ_ERR_INVALID   = -1,   /* NULL / inconsistent argument */
    TRQ_ERR_LAYOUT    = -2,   /* scene arrays violate the reference layout contract (bad index, cycle, ...) */
    TRQ_ERR_DEPTH     = -3,   /* interior depth > 31: the reference's 32-bit trail cannot represent it (Render.hh:140) */
    TRQ_ERR_CUDA      = -4,   /* a CUDA runtime call failed */
    TRQ_ERR_NOMEM     = -5,
    TRQ_ERR_NO_DEVICE = -6    /* no usable CUDA device: there is no CPU fallback */
} trq_status;

/* enum struct PrimitiveType  BVH.hh:6-8 */
enum { TRQ_SPHERE = 0, TRQ_SQUARE = 1, TRQ_CUBE = 2, TRQ_TRIANGLE = 3, TRQ_BVH = 4, TRQ_UNKNOW = 5 };

/* Mirrors struct Primitive (Render.hh:122-130) + element counts. Host pointers; arrays are
 * copied to the device by trq_scene_create and may be freed by the caller afterwards. */
typedef struct trq_scene_desc {
    const void*     sphereList;  uint32_t nSphere;   /* Sphere[nSphere],          272 B each */
    const void*     squareList;  uint32_t nSquare;   /* Square[nSquare],          272 B each */
    const void*     cubeList;    uint32_t nCube;     /* Cube[nCube],              240 B each */
    const void*     triList;     uint32_t nVert;     /* TriangleVertex[nVert],     32 B each */
    const uint32_t* idxList;     uint32_t nTri;      /* uint32[3*nTri]; leaf pIndex p -> idxList[3p..3p+2] */
    const void*     bvhList;     uint32_t nNode;     /* BVH[nNode], 64 B each, root at 0 */
} trq_scene_desc;

/* 32 B. Prefix-compatible with struct Ray (origin@0, direction@16); `tmax` is Scene::hit's
 * test_t (FLT_MAX for closest-hit of primary/bounce rays, light distance for shadow rays).
 * `direction` is used as given (Scene::hit never normalises; Ray's ctor already did), and no field is restricted:
 * every value has the oracle's answer, bit for bit. A -0.0 direction component gives 1/d = -inf; a NaN origin component is
 * dropped by every box test's fminf / fmaxf, so an all-NaN origin enters every box (at t = FLT_MIN, ties going right) and
 * visits the whole tree; a NaN tmax accepts leaves until one sets a finite range and otherwise ends as a miss; tmax <= 0 or
 * -inf misses; a direction need not be unit length (t is then in units of |direction|).
 * Spawned rays (trq_spawn_bounce / trq_spawn_shadow) use offset_ray, whose int(256 n) follows x86: truncation toward zero,
 * and INT32_MIN when n is NaN or |256 n| >= 2^31; the offset is added to the float's bits modulo 2^32. */
typedef struct trq_ray {
    float    ox, oy, oz, tmax;
    float    dx, dy, dz;
    uint32_t flags;              /* reserved, must be 0 */
} trq_ray;

#define TRQ_HIT_FLAG_HIT   1u
#define TRQ_HIT_FLAG_FRONT 2u    /* HitRecord::f  (HitRecord.hh:26-29) */

/* 32 B. All-zero on a miss. */
typedef struct trq_hit {
    float    t;                  /* HitRecord::t */
    uint32_t pType;              /* PrimitiveType of the winning leaf */
    uint32_t pIndex;             /* BVH::pIndex of the winning leaf */
    uint32_t leafNode;           /* index of the winning leaf in bvhList */
    float    u, v;               /* triangle: barycentrics u,v (Triangle.hh:61,65); others: HitRecord::uv */
    uint32_t material;           /* HitRecord::material */
    uint32_t flags;              /* TRQ_HIT_FLAG_* */
} trq_hit;

/* 16 B, opt-in (TRQ_HIT16): what a consumer needs to shade or to test occlusion, at half the bytes on every wire
 * (PCIe D2H, NVLink gather). id = 0xffffffff on a miss, else  front << 31 | pType << 28 | pIndex  (pIndex < 2^28);
 * t, u, v as in trq_hit. material and leafNode are not carried (material is a function of the primitive). */
typedef struct trq_hit16 {
    float    t;
    uint32_t id;
    float    u, v;
} trq_hit16;
#define TRQ_HIT16_MISS      0xffffffffu
#define TRQ_HIT16_FRONT(id) ((id) >> 31)
#define TRQ_HIT16_PTYPE(id) (((id) >> 28) & 7u)
#define TRQ_HIT16_PINDEX(id) ((id) & 0x0fffffffu)

/* 64 B. The HitRecord fields the query writes (for callers that shade). */
typedef struct trq_hit_record {
    uint32_t hit;
    float    t;
    float    p[3];
    float    gn[3];
    float    sn[3];
    float    uv[2];
    uint32_t front;
    uint32_t material;
    uint32_t pad;
} trq_hit_record;

typedef struct trq_scene_info_t {
    uint32_t nNode, nInterior, nLeaf;
    uint32_t maxDepth;           /* deepest interior level (root = 0); must be <= 31 */
    uint32_t nTri, nSphere, nSquare, nCube;
    uint64_t bytesReferenceLayout;   /* device bytes of the six arrays as uploaded */
    uint64_t bytesPacked;            /* device bytes of the derived traversal layout */
    int32_t  device;
    uint32_t topNodes;           /* interior nodes numbered breadth-first at the front of the packed array: the block the
                                    traversal kernel can stage in shared memory (top levels of the tree) */
} trq_scene_info_t;

/* trq_trace / trq_expand_hits flags */
#define TRQ_TRACE_ANY        0x1u   /* Scene::hit(..., any = true): first accepted hit ends the ray */
#define TRQ_HOST_PTRS        0x2u   /* rays / hits are HOST pointers: the library stages H2D / D2H
                                       (chunked, overlapped with tracing) and returns after completion */
#define TRQ_KERNEL_REFLAYOUT 0x4u   /* run the 1:1 transcription over the reference-layout buffers
                                       (correctness anchor / naive baseline) instead of the packed kernel */
#define TRQ_SORT_RAYS        0x8u   /* hint: the batch is incoherent; the library orders the work queue by
                                       (origin cell, direction octant) first. Results are identical either way.
                                       Without the hint, a scene whose packed tree exceeds twice the L2 cache has its
                                       batches of >= 2^20 rays examined (one streaming pass) and ordered when fewer than
                                       half of the neighbouring rays share a cell and octant. */
#define TRQ_NO_SORT          0x40u  /* never order the work queue (switches the automatic mode off for this call) */

#define TRQ_HIT16            0x20u  /* `hits` is trq_hit16[n] (16-byte aligned) instead of trq_hit[n] */

#define TRQ_HOST_ASYNC       0x10u  /* with TRQ_HOST_PTRS: return as soon as the copies and kernels are queued; the host
                                       buffers must stay valid (and should be pinned) until trq_host_sync() returns.
                                       Consecutive calls then overlap: the next batch's H2D runs under this one's D2H. */

/* trq_scene_rebuild flags (with TRQ_HOST_PTRS) */
#define TRQ_BUILD_MORTON     0x80u  /* build the new topology with the Morton builder (trq_bvh_build_tree_morton_device) */

typedef struct trq_scene trq_scene;

int  trq_version(void);
const char* trq_last_error_string(void);
int  trq_device_count(void);

/* Uploads the six arrays to `device`, validates the tree (indices in range, every node the root
 * reaches well linked, interior depth <= 31) and derives the packed traversal layout on the device.
 * Nodes the root does not reach are kept but never read: not by a trace, not by a refit. */
int  trq_scene_create(const trq_scene_desc* desc, int device, trq_scene** out);
/* The same for a scene that already lives on the GPU: every array of `desc` is a DEVICE pointer on `device` (for
 * example bvhList from trq_bvh_build_tree_device). The arrays are copied device to device; validation and numbering
 * run as kernels, so no array crosses PCIe (128 bytes of counters come back). Same checks and same packed layout as
 * trq_scene_create, with one difference: EVERY node of bvhList must be reachable from the root. */
int  trq_scene_create_device(const trq_scene_desc* desc, int device, trq_scene** out);

/* Refit after the vertices moved (animated meshes): same topology, new boxes. Triangle leaf boxes are recomputed from
 * the new vertices (min / max of the three, AAPLRenderer.mm:575-589), interior boxes bottom-up as the union of their
 * children (AABB::make, BVH.hh:229-231), the packed layout is derived again; all on the device. Only nodes the root reaches
 * are refit (a one-leaf scene's root leaf included). triList holds the
 * scene's nVert vertices: a device pointer, or a host pointer with TRQ_HOST_PTRS. Synchronous: waits for traces in
 * flight, returns when the scene is ready for the next trq_trace. */
int  trq_scene_update_vertices(trq_scene* scene, const void* triList, uint32_t nVert, uint32_t flags);

/* Refit after primitives moved (animated spheres, squares, cubes and meshes): same topology, new boxes. A scene update
 * is trq_scene_update_vertices for every leaf type.
 *   changes    each non-NULL sphereList / squareList / cubeList / triList replaces that array of the scene whole; its count
 *              must equal the scene's list count (the nSphere / nSquare / nCube / nVert the scene was created with, not
 *              its leaf counts). A NULL pointer with count 0 keeps that array. idxList and bvhList must be NULL with count
 *              0: they would change the topology. All arrays are device pointers on the scene's device, or all are host
 *              pointers with TRQ_HOST_PTRS.
 *   leaves     every leaf the root reaches whose primitive type was replaced gets new bBOX mini / maxi. A sphere, square
 *              or cube leaf gets, bit for bit, the box trq_bvh_build_node(list[pIndex].box.mini, .maxi, list[pIndex].model,
 *              pType, pIndex) writes, with `box` the record's boundingBOX (Sphere, Square) or box (Cube)
 *              (AAPLRenderer.mm:454-468). A triangle leaf gets what trq_scene_update_vertices gives it.
 *   kept       parent, left, right, axis, pType, pIndex and the padding words of every node, byte for byte. Leaves the root
 *              does not reach and leaves of unknown pType keep their boxes.
 *   interior   the interior nodes the root reaches are refit bottom-up as unions of their children, as in
 *              trq_scene_update_vertices; a one-leaf scene's root leaf is refit like any other leaf.
 *   derived    the packed layout (sphere centre, radius and material; square ranges, axes and material; interior nodes; the
 *              top-of-tree block) and the root box are derived again. Everything that reads the lists sees the new records:
 *              traces (the reference-layout kernel and cubes included), trq_expand_hits, and the bounce and shadow spawns,
 *              so replacing squareList moves the lights trq_spawn_shadow samples even where the squares have no leaves.
 *   unchanged  trq_scene_info, the leaf types the traversal kernels are specialised for, the launch configurations and a
 *              configuration chosen with trq_scene_set_kernel_config.
 *   failure    TRQ_ERR_INVALID (NULL scene or changes, a count mismatch, a non-NULL idxList / bvhList, a NULL array with a
 *              non-zero count), TRQ_ERR_NOMEM (no scratch): the scene is exactly as before.
 * Synchronous: waits for traces in flight, returns when the scene is ready for the next trq_trace. */
int  trq_scene_update_primitives(trq_scene* scene, const trq_scene_desc* changes, uint32_t flags);

/* Rebuild: a new topology from the scene's current geometry, on the device, in place -- for motion a refit cannot follow
 * (a refit tree's boxes stretch and overlap as the geometry moves, and every ray pays for it). triList: the scene's nVert
 * new vertices (a device pointer, or a host pointer with TRQ_HOST_PTRS), or NULL (nVert 0) to keep the current ones.
 *   leaf list  every leaf the root reaches, in ascending bvhList index order. For a tree trq_bvh_build_tree(_gpu/_device)
 *              made these are nodes 1..n in list order, so rebuilding an unchanged scene reproduces its tree byte for byte.
 *   leaves     a triangle leaf keeps its pIndex; its box is what trq_bvh_build_nodes_triangles gives for that triangle
 *              from the current vertices (std::min / std::max of the three, then BVH::buildNode with the identity). Every
 *              other leaf (sphere, square, cube, unknown pType) keeps pType, pIndex and box: to move those primitives,
 *              move them with trq_scene_update_primitives first. All other fields are zero, as trq_bvh_build_node writes them.
 *   tree       what trq_bvh_build_tree_gpu makes from that leaf list (the host builder's tree except where its std::sort
 *              fallback meets equal or NaN keys, see there); nNode becomes 2n - 1, so a scene whose bvhList had
 *              unreachable nodes shrinks.
 *   state      afterwards the scene is indistinguishable from one trq_scene_create_device made from the new tree: info
 *              (maxDepth, topNodes, nNode, bytesReferenceLayout, ...), packed arrays, top-of-tree block, and every launch
 *              configuration's usability and staged node count. A configuration chosen with trq_scene_set_kernel_config
 *              is kept if it is still usable; otherwise the scene uses the automatic choice for the new tree.
 *   builder    with TRQ_BUILD_MORTON in flags, the tree over the same leaf list is trq_bvh_build_tree_morton_device's
 *              instead: much faster to build, usually slower to trace, never deeper than 31. Everything else is as above.
 *   failure    TRQ_ERR_DEPTH (new interior depth > 31; the message gives it), TRQ_ERR_NOMEM, TRQ_ERR_INVALID (nVert other
 *              than the scene's): the scene is exactly as before, vertices included.
 * Synchronous: waits for work in flight on the device, returns when the scene is ready for the next trq_trace. Hits traced
 * before a rebuild name leaves (trq_hit.leafNode) by the OLD numbering. trq_scene_update_vertices refits the new tree. */
int  trq_scene_rebuild(trq_scene* scene, const void* triList, uint32_t nVert, uint32_t flags);

/* Copies the scene's node array (trq_scene_info_t.nNode nodes, 64 B each) to `out`: a device pointer on the scene's
 * device, or a host pointer with TRQ_HOST_PTRS. Synchronous. */
int  trq_scene_copy_bvh(const trq_scene* scene, void* out, uint32_t flags);

int  trq_scene_destroy(trq_scene* scene);

/* Scene arrays and builder scratch come from a per-device memory pool that keeps what it is given back (so that
 * destroy + create of a similar scene, or a rebuild every frame, costs no cudaMalloc). This returns the cached memory of
 * `device` to the driver. */
int  trq_device_trim(int device);
int  trq_scene_info(const trq_scene* scene, trq_scene_info_t* info);

/* Launch configurations of the traversal kernel (tuning knob; results are identical in all of them). A configuration is
 * "CTA size x resident CTAs per SM", with or without the top levels of the tree staged in shared memory by a TMA bulk
 * copy (names end in "true" / "false"). cfg < 0 selects the library's choice for this scene. TRQ_CFG=<n> in the
 * environment overrides every scene (experiments). topNodesStaged (optional): how many interior nodes that
 * configuration keeps in shared memory for this scene. */
int  trq_kernel_config_count(void);
const char* trq_kernel_config_name(int cfg);
int  trq_scene_set_kernel_config(trq_scene* scene, int cfg, uint32_t* topNodesStaged);
/* The configuration this scene's traces use now (index into trq_kernel_config_name), or -1 for a NULL scene. */
int  trq_scene_kernel_config(const trq_scene* scene);

/* Scene::hit for n rays. Device pointers unless TRQ_HOST_PTRS; asynchronous on `stream`
 * (a cudaStream_t, NULL = default stream) for device pointers. Re-entrant across streams and host threads, and
 * capturable into CUDA graphs. Work-queue heads: a launch captured into a graph allocates, zeroes and frees a head of its
 * own at every replay, so graphs captured at any time may be replayed concurrently with each other and with eager
 * calls. Eager launches of a scene take heads from a ring of 4096 that the kernel re-arms: launch k and launch k + 4096
 * of one scene share a head and must not run at the same time, so with many streams keep fewer than 4096 launches of a
 * scene issued beside a long-running one (a single stream always satisfies this).
 * A batch of more than 2^31 rays is traced as consecutive launches of at most 2^31 rays each.
 * `hits` is trq_hit[n], or trq_hit16[n] with TRQ_HIT16. Device rays / hits must be aligned to their record size
 * (32 bytes; 16 for trq_hit16): every record is moved with one access. */
int  trq_trace(trq_scene* scene, const trq_ray* rays, uint64_t n, uint32_t flags,
               void* hits, void* stream);

/* Waits for every TRQ_HOST_ASYNC call issued on this scene. */
int  trq_host_sync(trq_scene* scene);

/* Fills HitRecord fields p, gn, sn, uv, f, material for hits produced by trq_trace. */
int  trq_expand_hits(trq_scene* scene, const trq_ray* rays, const trq_hit* hits, uint64_t n,
                     uint32_t flags, trq_hit_record* records, void* stream);

/* ---- wavefront callers (the producers either side of the query; device pointers only) ----------------------
 * With these a cast -> trace -> spawn -> trace ... wavefront stays on the GPU: spawn compacts the surviving rays
 * into `out` with one atomic per warp and leaves their number in device memory (*d_count), which
 * trq_trace_indirect and the next spawn read on the device (no host round trip).
 * Overlap: the outputs of a call must not share memory with its inputs. A spawn zeroes *d_count on the stream before its
 * kernel reads *d_n, so d_count == d_n spawns nothing; out / srcIndex overlapping rays / hits (or trq_trace_indirect's
 * hits overlapping rays / d_count) is a race whose result is undefined. */

/* Arguments of MakeCamera (RT_Metal/Tracer/Tracer.mm:87-125); vfov in radians, as the reference passes it. */
typedef struct trq_camera {
    float lookFrom[3], lookAt[3], viewUp[3];
    float vfov, aspect, aperture, focus_dist;
} trq_camera;

/* castRay for every pixel of a W x H image (Camera.hh:59-69 with s = x/W, t = y/H, Render.metal:523-527):
 * rays[y*W + x], tmax = FLT_MAX. Only aperture 0 (the reference's prepareCamera, Tracer.mm:380). */
int  trq_cast_rays(trq_scene* scene, const trq_camera* camera, uint32_t W, uint32_t H, trq_ray* rays, void* stream);

/* Scene::hit with the batch size read from device memory: traces min(*d_count, capacity) rays. One launch covers the
 * whole capacity, so a capacity above 2^31 is refused (TRQ_ERR_INVALID) whatever *d_count holds. */
int  trq_trace_indirect(trq_scene* scene, const trq_ray* rays, const uint64_t* d_count, uint64_t capacity,
                        uint32_t flags, trq_hit* hits, void* stream);

/* Diffuse bounce of tracePath (Render.metal:447-475): for every hit i < n (n clamped to *d_n when d_n != NULL):
 * PCG32(seedBase + i, 1) -> uu; origin = offset_ray(p, sn); direction = normalize(stw * CosineSampleHemisphere(uu));
 * tmax = FLT_MAX. out needs room for n rays; srcIndex (optional) receives i per output ray; *d_count the total. */
int  trq_spawn_bounce(trq_scene* scene, const trq_ray* rays, const trq_hit* hits, uint64_t n, const uint64_t* d_n,
                      uint64_t seedBase, trq_ray* out, uint32_t* srcIndex, uint64_t* d_count, void* stream);

/* NEE shadow ray of traceMIS (Render.metal:313-337): toward a point sampled (Square::sample, Square.hh:40-58) on
 * squareList[lightA] or squareList[lightB] (picked by random() < 0.5), tmax = distance; trace with TRQ_TRACE_ANY. */
int  trq_spawn_shadow(trq_scene* scene, const trq_ray* rays, const trq_hit* hits, uint64_t n, const uint64_t* d_n,
                      uint64_t seedBase, uint32_t lightA, uint32_t lightB, trq_ray* out, uint32_t* srcIndex,
                      uint64_t* d_count, void* stream);

/* The two spawns drawing from the reference's per-pixel RNG state texture (row f-4: RGBA32Uint, 4 x uint32 per pixel).
 * The array is kept in the layout exRNG writes at kernel exit (Render.hh:109-120, Render.metal:545-556):
 * {state >> 32, state, inc >> 32, inc}. Ray i belongs to pixel pixelOf[i] (NULL: i); its PCG32 stream is loaded from
 * rngState[4 * pixel], advanced by the draws and stored back in the same layout, so the next wave continues it.
 * srcIndex[k] receives the PIXEL of output ray k: pass it as pixelOf of the next wave. rngState == NULL behaves like the
 * calls above (PCG32(seedBase + i, 1)). Two rays of one batch must not share a pixel.
 * Frame boundary: the reference's toRNG at kernel ENTRY (Render.hh:96-107) brace-initialises pcg32_t {state, inc}
 * (Random.hh:6-12) with (inc, state), i.e. it reads the words exRNG stored as the state as the increment and vice
 * versa -- the halves of a texel trade places once per frame. trq_rng_frame_begin applies exactly that (in place,
 * once per frame, before the first wave); with it the array evolves like the reference's texture frame after frame. */
int  trq_rng_frame_begin(trq_scene* scene, uint32_t* rngState, uint64_t nPixels, void* stream);
int  trq_spawn_bounce_rng(trq_scene* scene, const trq_ray* rays, const trq_hit* hits, uint64_t n, const uint64_t* d_n,
                          uint64_t seedBase, const uint32_t* pixelOf, uint32_t* rngState, trq_ray* out, uint32_t* srcIndex,
                          uint64_t* d_count, void* stream);
int  trq_spawn_shadow_rng(trq_scene* scene, const trq_ray* rays, const trq_hit* hits, uint64_t n, const uint64_t* d_n,
                          uint64_t seedBase, const uint32_t* pixelOf, uint32_t* rngState, uint32_t lightA, uint32_t lightB,
                          trq_ray* out, uint32_t* srcIndex, uint64_t* d_count, void* stream);

/* ---- multi-GPU in one process (the reference's host is a single application) -----------------------------------
 * One scene per device, created from the same host arrays; host rays are cut into contiguous ranges
 * [k*n/R, (k+1)*n/R) (trq_mgpu_shard) and every range is staged and traced on its own device at the same time; the
 * hits land in the caller's array. No collective is involved (SURVEY.md section 8e). devices == NULL: devices 0..n-1;
 * nDevices <= 0: every visible device. trq_mgpu_scene gives the k-th scene for device-pointer work on that GPU. */
typedef struct trq_mgpu trq_mgpu;
int  trq_mgpu_create(const trq_scene_desc* desc, const int* devices, int nDevices, trq_mgpu** out);
int  trq_mgpu_device_count(const trq_mgpu* m);
trq_scene* trq_mgpu_scene(trq_mgpu* m, int k);
int  trq_mgpu_shard(const trq_mgpu* m, uint64_t n, int k, uint64_t* lo, uint64_t* hi);
int  trq_mgpu_trace(trq_mgpu* m, const trq_ray* rays, uint64_t n, uint32_t flags, void* hits /* trq_hit[n], or trq_hit16[n] with TRQ_HIT16 */);
int  trq_mgpu_destroy(trq_mgpu* m);

/* ---- multi-GPU: hit gather through NVLink peer memory (one process per GPU, one node) -----------------------
 * Rays shard across ranks with no collective (SURVEY.md section 8e). A consumer that wants EVERY rank's hits whole
 * (the all-gather of trq_hit[N/R] of section 8e) gets them while the traversal is still running: the trace kernel
 * counts finished records per tile of 2^TRQ_GATHER_TILE_SHIFT records (environment, 8..16, default 11: 2048 records),
 * and a sender kernel that shares the SMs with it ships every complete tile into slot [rank] of every other rank's
 * buffer over NVLink -- compute and all-gather overlap tile by tile -- then publishes (count, step) with system-scope
 * release stores. No NCCL call. The sender is by default the TMA one (bulk copies through 24 KB of shared memory, in
 * 12 KB chunks). The LSU sender (coalesced 16-byte loads and stores, no shared memory) runs instead when
 * TRQ_GATHER_TMA=0, or when those 24 KB do not fit in the SM beside the resident trace CTAs, which happens for
 * deep trees (a larger far-child stack per ray). Both give the same bytes.
 *   1. every rank: trq_gather_create -> 64-byte handle; exchange the handles (any transport, e.g. MPI /
 *      torch.distributed all_gather) into a world*64-byte array in rank order; trq_gather_connect.
 *   2. per step: trq_trace_gather(rays of this rank) then trq_gather_wait -> hitsAll, counts[r]; rank r's records
 *      start at byte r * capacity * 32 of hitsAll and are trq_hit, or trq_hit16 when the step was traced with
 *      TRQ_HIT16 (same slot stride). Both calls are asynchronous on `stream`; the buffers rotate through three phases,
 *      so the result of step k stays valid until this rank's trq_trace_gather for step k+2 EXECUTES (a peer cannot
 *      reuse the phase before it has seen this rank finish step k+2). Every rank must call both every step.
 *   3. all ranks synchronise (barrier) before any of them calls trq_gather_destroy.
 * trq_gather_status (after synchronising the stream) reports a peer that never published (timeout 10 s,
 * TRQ_GATHER_TIMEOUT_MS) instead of hanging the GPU.
 * A step is one kernel launch: the capacity is at most 2^31 rays (trq_gather_create refuses more), and trq_trace_gather
 * refuses n above the capacity. */
typedef struct trq_gather trq_gather;
#define TRQ_GATHER_HANDLE_BYTES 64
int  trq_gather_create(trq_scene* scene, uint32_t rank, uint32_t world, uint64_t capacity, trq_gather** out,
                       void* handle /* TRQ_GATHER_HANDLE_BYTES */);
int  trq_gather_connect(trq_gather* g, const void* handles /* world * TRQ_GATHER_HANDLE_BYTES, rank order */);
int  trq_trace_gather(trq_scene* scene, trq_gather* g, const trq_ray* rays, uint64_t n, uint32_t flags, void* stream);
int  trq_gather_wait(trq_gather* g, void* stream, const void** hitsAll, const uint64_t** counts);
int  trq_gather_status(trq_gather* g);
int  trq_gather_destroy(trq_gather* g);

/* Per-kernel timing for roofline reports: when enabled, every device-pointer trq_trace records CUDA
 * events (on the caller's stream) around the traversal kernel (with its ordering passes, if any) and
 * around what follows it -- the resolve pass of TRQ_KERNEL_REFLAYOUT; the packed kernel finishes its own
 * records, so resolveKernelMs is 0 for it. A trace that follows another trace of the same tree on its stream
 * starts under that one's tail (programmatic dependent launch), and an event between the two would make it wait:
 * such a launch is timed by the kernel itself (%globaltimer at its first CTA's start and its last CTA's exit), and
 * these launches count with the time during which at least one of them ran. trq_profile_read waits for the
 * launches and returns the SUMS over the launches since the last read (at most the 64 most recent) and resets.
 * Not for TRQ_HOST_PTRS calls. */
int  trq_profile_enable(trq_scene* scene, int on);
int  trq_profile_read(trq_scene* scene, uint32_t* nLaunches, float* traceKernelMs, float* resolveKernelMs);

/* Read bandwidth of the memory system as this library's kernels see it (16-byte loads that bypass L1, all SMs, best of
 * five): which = 0 -> 32 MB working set (L2), which = 1 -> 2 GB working set (HBM). For the roofline report. */
int  trq_probe_bandwidth(int device, int which, double* gbs);

/* Number of kernel launches issued by this library in this process (bench evidence). */
uint64_t trq_launch_count(void);

/* ---- host side: reference scene preparation, restated (BVH.hh:246-314) ------------------- */

/* BVH::buildNode: world AABB of the 8 corners of [box_min, box_max] under the column-major
 * model matrix; writes one 64-B leaf. model == NULL means identity. */
int  trq_bvh_build_node(const float box_min[3], const float box_max[3], const float model[16],
                        int32_t pType, uint32_t pIndex, void* node_out);

/* Per-triangle leaves as AAPLRenderer.mm:575-589 does: box = min/max of the 3 vertices,
 * identity model, pType = Triangle, pIndex = pIndexBase + i. Writes nTri 64-B nodes. */
int  trq_bvh_build_nodes_triangles(const void* triList, const uint32_t* idxList, uint32_t nTri,
                                   uint32_t pIndexBase, void* nodes_out);

/* The same leaves built on the GPU, bit for bit (NaN, signed zeros and infinities included): device pointers on `device`,
 * asynchronous on `stream` (a cudaStream_t, NULL = default stream). nTri == 0 is a no-op. With the vertices already on
 * the GPU, this + trq_bvh_build_tree_device + trq_scene_create_device make a scene without the host touching an array. */
int  trq_bvh_build_nodes_triangles_device(const void* d_triList, const uint32_t* d_idxList, uint32_t nTri,
                                          uint32_t pIndexBase, void* d_nodes_out, int device, void* stream);

/* BVH::buildNode on the GPU for n spheres / squares / cubes (pType TRQ_SPHERE / TRQ_SQUARE / TRQ_CUBE; anything else is
 * TRQ_ERR_INVALID) given in their reference layout (272 / 272 / 240 B): leaf k = trq_bvh_build_node(list[k].box.mini,
 * list[k].box.maxi, list[k].model, pType, pIndexBase + k), bit for bit -- the box is boundingBOX for Sphere and Square,
 * box for Cube (AAPLRenderer.mm:454-468). Device pointers, asynchronous on `stream`; n == 0 is a no-op. */
int  trq_bvh_build_nodes_device(int32_t pType, const void* d_list, uint32_t n, uint32_t pIndexBase,
                                void* d_nodes_out, int device, void* stream);

/* BVH::buildTree: on entry bvhList[0..nLeaves) are leaves (capacity >= 2*nLeaves-1 nodes);
 * on return the array holds the reference's final order: root at 0, leaves at 1..nLeaves,
 * interiors after, parent/left/right = final indices. Sequential variant (deterministic).
 * *maxDepthOut = deepest interior level (root = 0). Interior depth above 31 returns TRQ_ERR_DEPTH
 * with the complete tree in bvhList and its true depth in *maxDepthOut. */
int  trq_bvh_build_tree(void* bvhList, uint32_t nLeaves, uint32_t* nNodeOut, uint32_t* maxDepthOut);

/* The same build on the GPU (level-synchronous binned SAH, kernels/bvh_build.cuh): same arguments (HOST array in
 * and out), same node array byte for byte -- splits, child order, numbering, boxes -- except where the reference's
 * std::sort fallback sorts equal or NaN keys, whose order std::sort leaves unspecified: three or more primitives
 * sharing one centroid, or a node spanning an infinite centroid extent (a leaf side at +inf, centroids near
 * +-FLT_MAX) in which two keys on the split axis are equal or NaN. The GPU sorts such a node stably, NaN last.
 * Interior depth above 31 returns TRQ_ERR_DEPTH with the complete tree and its true depth, as trq_bvh_build_tree
 * does. TRQ_ERR_NO_DEVICE without a GPU (use the host builder). */
int  trq_bvh_build_tree_gpu(void* bvhList, uint32_t nLeaves, int device, uint32_t* nNodeOut, uint32_t* maxDepthOut);

/* The same build with the array in DEVICE memory on `device` (leaves in d_bvhList[0..nLeaves), capacity 2*nLeaves-1
 * nodes; the result replaces them): build -> trq_scene_create_device without the tree ever visiting the host.
 * Interior depth above 31 returns TRQ_ERR_DEPTH with the complete tree in d_bvhList and its true depth. */
int  trq_bvh_build_tree_device(void* d_bvhList, uint32_t nLeaves, int device, uint32_t* nNodeOut, uint32_t* maxDepthOut);

/* The Morton-order (LBVH) builder: a tree in the same node format and layout (root at 0, leaves at 1..nLeaves in list
 * order, interiors after, parent/left/right final indices), built in a fraction of the SAH builder's time at some cost in
 * trace speed. It never returns TRQ_ERR_DEPTH: every tree it builds has interior depth <= 31. Its tree, for n leaves:
 *   centroid   AABB::centroid (AABB.hh:22-25) of each leaf box: mini + (maxi - mini) / 2.
 *   quantise   per axis, strict fp32: lo / hi = min / max of the FINITE centroid components on that axis. NaN and +inf
 *              give 2^21 - 1, -inf gives 0. Where the axis has no finite component, or hi - lo is not (finite and > 0),
 *              every finite component gives 0. Otherwise q = min(2^21 - 1, floor(((c - lo) / (hi - lo)) * 2^21)), each
 *              operation rounded to nearest, in that order.
 *   code       63 bits: bit 3i+2 is bit i of qx, bit 3i+1 of qy, bit 3i of qz.
 *   order      leaves sorted by (code, list position).
 *   topology   top-down; a node at interior depth d (root 0) over sorted positions [a, b], m = b - a + 1: the left child
 *              gets floor(m / 2) leaves if code[a] == code[b], else the positions whose code has clear the highest bit in
 *              which code[a] and code[b] differ. That size is clamped into [m - 2^(31-d), 2^(31-d)] intersected with
 *              [1, m - 1], which bounds the depth at 31 and changes nothing where the tree is shallow enough already.
 *   numbering  the interior node splitting between sorted positions g and g + 1 is node n + 1 + g if g is below the root's
 *              gap, else n + g. n == 1: the lone leaf is node 0 with parent 0.
 *   fields     axis = dimension of the highest bit in which the node's two end codes differ (0 if equal); pType TRQ_BVH,
 *              pIndex 0, padding 0; box = union of the child boxes (fminf / fmaxf). Leaves keep every field but parent.
 * Host restatement: bvhList as for trq_bvh_build_tree (capacity 2*nLeaves-1 nodes). TRQ_ERR_INVALID for an empty list or
 * more than 0x3fffffff leaves. */
int  trq_bvh_build_tree_morton(void* bvhList, uint32_t nLeaves, uint32_t* nNodeOut, uint32_t* maxDepthOut);

/* The same tree, byte for byte, built on `device` with the array in DEVICE memory (as trq_bvh_build_tree_device: leaves
 * in d_bvhList[0..nLeaves), capacity 2*nLeaves-1 nodes, the result replaces them). Synchronous, on the legacy default
 * stream. TRQ_ERR_INVALID as the host restatement, TRQ_ERR_NO_DEVICE without a GPU. */
int  trq_bvh_build_tree_morton_device(void* d_bvhList, uint32_t nLeaves, int device, uint32_t* nNodeOut, uint32_t* maxDepthOut);

#ifdef __cplusplus
}
#endif
#endif /* TRACER_RQ_H */
