// tracer_b200/csrc/trq_api.cu -- implementation of the C-ABI in include/tracer_rq.h.
//
// Host side of the drop-in boundary: it takes the six reference-layout arrays exactly as
// AAPLRenderer.mm:614-624,712-720 hands them to Metal (struct Primitive, Render.hh:122-130),
// uploads them, derives the packed traversal layout ON THE DEVICE (pack_scene_kernel), and runs
// batches of Scene::hit (Render.hh:135-252) as CUDA kernels. No CPU fallback exists: without a
// device every compute entry point returns TRQ_ERR_NO_DEVICE.

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <utility>
#include <vector>

#include "../../include/tracer_rq.h"
#include "host/error.h"
#include "host/gpu_build.h"
#include "host/layout.h"
#include "host/scratch.h"
#include "kernels/plan_scene.cuh"
#include "kernels/trace_kernels.cuh"

using namespace trq;

namespace {

std::atomic<uint64_t> g_launches{0};

}  // namespace

namespace trq { void note_launches(uint64_t n) { g_launches += n; } }   // other translation units (GPU builder)



namespace {

#define TRQ_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess)                                                                  \
            return trq::fail(TRQ_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// developer instrumentation (tools/build_variant.sh timing -DTRQ_CREATE_TIMING): wall time of the stages of scene creation
#ifdef TRQ_CREATE_TIMING
struct StageTimer {
    std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
    void lap(const char* what) {
        cudaDeviceSynchronize();
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "  [create] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t).count());
        t = now;
    }
};
#define TRQ_LAP(timer, what) (timer).lap(what)
#else
struct StageTimer {};
#define TRQ_LAP(timer, what) ((void)(timer))
#endif

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; }
        ok = (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

constexpr int kQueueRing = 4096;           // queue heads of eager launches, handed out round-robin; each is zero between launches
                                           // (the kernel's last CTA re-arms it). Launch k and launch k + 4096 share one: they
                                           // must not run at the same time (trq_trace in include/tracer_rq.h)
constexpr int kStageBufs = 4;
constexpr int kProfRing = 64;
constexpr size_t kSmemPerSM = 228u * 1024u, kSmemPerBlockMax = 227u * 1024u, kSmemBlockReserve = 1024u;
constexpr size_t kSmemDynamicMax = kSmemPerBlockMax - 1024u;   // dynamic part: the kernel also has a few static bytes (mbarrier)

// Launch configurations of trace_packed_kernel: CTA size x resident CTAs per SM, with or without the top of the tree
// staged in shared memory. [any][record format] -> kernel.
struct KernelCfg {
    int block, minb;
    bool top;
    const void* fn[3][2][2];      // [leaf types present: LEAVES_*][any][record format]
    const char* name;
};
#define TRQ_CFG_FN(B, M, T, R)                                                                                \
      { { (const void*)trace_packed_kernel<false, OUT_HIT32, B, M, T, R>, (const void*)trace_packed_kernel<false, OUT_HIT16, B, M, T, R> }, \
        { (const void*)trace_packed_kernel<true, OUT_HIT32, B, M, T, R>, (const void*)trace_packed_kernel<true, OUT_HIT16, B, M, T, R> } }
#define TRQ_CFG(B, M, T) { B, M, T, { TRQ_CFG_FN(B, M, T, LEAVES_ALL), TRQ_CFG_FN(B, M, T, LEAVES_TRI_SPHERE), TRQ_CFG_FN(B, M, T, LEAVES_TRI) }, #B "x" #M " top=" #T }
const KernelCfg kCfgs[] = {
    TRQ_CFG(256, 5, false),       // 0: five CTAs of 256 threads per SM, every node from L1 / L2 (large scenes)
    TRQ_CFG(1024, 1, true),       // 1: one CTA of 1024 threads per SM sharing one TMA-staged copy of the top levels (small trees)
#ifdef TRQ_EXTRA_CFGS
    TRQ_EXTRA_CFGS
#endif
};
constexpr int kNumCfgs = (int)(sizeof(kCfgs) / sizeof(kCfgs[0]));
#ifndef TRQ_DEFAULT_CHUNK_RAYS
#define TRQ_DEFAULT_CHUNK_RAYS (512ll << 10)
#endif
// Largest batch one kernel launch takes (the kernels keep a 32-bit ray index per lane); trq_trace splits larger ones.
// Smaller values build test variants that exercise the split on small batches.
#ifndef TRQ_MAX_RAYS_PER_LAUNCH
#define TRQ_MAX_RAYS_PER_LAUNCH (1ull << 31)
#endif

// Scene arrays come from the per-device pool that keeps its memory (host/scratch.h): a scene created after another one of
// similar size was destroyed gets its memory back without a cudaMalloc (about 1 ms each for these sizes: 15 of the 22 ms
// of a 1 M-triangle trq_scene_create_device before). trq_device_trim() hands cached memory back to the driver.
cudaError_t pool_malloc(void** p, size_t bytes) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    cudaMemPool_t pool = trq::scratch_pool(dev);
    return pool ? cudaMallocFromPoolAsync(p, bytes, pool, nullptr) : cudaMalloc(p, bytes);
}
void pool_free(void* p) { if (p) cudaFreeAsync(p, nullptr); }

// One launch configuration for one tree: staged top-of-tree nodes, dynamic shared memory, resident CTAs per SM [any][format]
struct CfgState { uint32_t topCount = 0, stackDepth = 0; size_t smem = 0; int blocksPerSM[2][2] = {}; bool usable = false; };

// The records a rebuild keeps: device copies of the reference-layout lists (struct Primitive) and their lengths.
struct SceneRecords {
    RefSphere* spheres = nullptr; RefSquare* squares = nullptr; RefCube* cubes = nullptr; RefVertex* verts = nullptr; uint32_t* idx = nullptr;
    uint32_t nSphere = 0, nSquare = 0, nCube = 0, nVert = 0, nTri = 0;   // records in the lists (info counts leaves)
    void release() { pool_free(spheres); pool_free(squares); pool_free(cubes); pool_free(verts); pool_free(idx); *this = SceneRecords(); }
};

// The tree and everything derived from it: what a rebuild replaces whole.
struct PackedTree {
    RefBVH*   bvh = nullptr;
    uint32_t* ref = nullptr;      // packed reference of every bvhList node (kept for refits)
    float4 *nodes = nullptr, *tris = nullptr, *sph = nullptr, *sq = nullptr, *triN = nullptr, *topSoA = nullptr;   // packed_layout.cuh
    trq_scene_info_t info{};
    uint32_t nSqLeaf = 0;         // square leaves (info.nSquare counts records)
    uint32_t rootRef = 0, stackDepth = 1;
    float rootMin[3] = {}, rootMax[3] = {};
    bool largeTree = false;       // packed tree > 2 x L2: incoherent batches are worth ordering (automatic TRQ_SORT_RAYS)
    int leaves = 0;               // LEAVES_*: which leaf types the tree has (selects the kernels without the other types' code)
    uint32_t maxPIndex = 0;       // largest leaf pIndex (trq_hit16 packs it into 28 bits)
    CfgState cfg[kNumCfgs];
    int autoCfg = 0;
    void release() {
        pool_free(bvh); pool_free(ref); pool_free(nodes); pool_free(tris); pool_free(sph); pool_free(sq); pool_free(triN); pool_free(topSoA);
        *this = PackedTree();
    }
};

}  // namespace

struct trq_scene {
    int device = 0;
    int numSMs = 0;
    SceneRecords rec;
    PackedTree tree;
    int defaultCfg = 0;
    bool userCfg = false;         // defaultCfg was chosen with trq_scene_set_kernel_config (kept by a rebuild while usable)
    // stream-ordered scratch for TRQ_SORT_RAYS: a private pool that keeps its memory across synchronisations
    // (the device's default pool hands it back at every sync and re-maps 64 MB on the next sorted launch)
    cudaMemPool_t scratchPool = nullptr;     // the per-device pool (not owned); also holds the queue heads of captured launches
    // ray-queue heads of eager launches
    QueueHead* d_queues = nullptr;
    std::atomic<uint32_t> queueNext{0};
    // staging for TRQ_HOST_PTRS
    std::mutex stageMutex;
    uint64_t stageCap = 0;
    trq_ray* d_stageRays[kStageBufs] = {};
    trq_hit* d_stageHits[kStageBufs] = {};
    cudaStream_t stageStream[kStageBufs] = {};   // one stream per staging buffer: copy in, trace, copy out in stream order
    bool stageReady = false;
    uint64_t stageSeq = 0;        // chunks ever staged (ring position)
    // optional per-kernel timing (trq_profile_enable): events around the trace and resolve kernels; an early launch (below)
    // is timed by the kernel itself instead, since an event recorded between two kernels makes the second wait for the first
    std::mutex profMutex;
    bool profile = false;
    cudaEvent_t evProf[kProfRing][3] = {};
    unsigned long long* d_profStamps = nullptr;   // [kProfRing][2]: {start, end} of an early launch (TraceParams::timing)
    bool profByKernel[kProfRing] = {};
    uint32_t profHead = 0, profCount = 0;
    // A trace has been launched on the tree as it now is (cleared by a refit or a rebuild): the next trace may be an early
    // launch, one whose CTAs start while the previous kernel on its stream is still running (launch_trace).
    std::atomic<bool> treeTraced{false};
    uint32_t tailSeq = 0;         // TRQ_TAIL_TIMELINE builds: launches since trq_debug_tail's reset
    // Scratch in which early launches park the records they finish before their wait (TraceParams::park): two halves, taken
    // in turn by the early launches on one stream (the first that asks). Two launches that overlap are consecutive on their
    // stream, so they never share a half; early launches on other streams do without.
    std::mutex parkMutex;
    float4* d_park = nullptr;
    uint32_t* d_parkRunning = nullptr;   // [2]: one word per half (TraceParams::parkRunning)
    size_t parkHalf = 0;
    cudaStream_t parkStream = nullptr;
    bool parkBound = false;
    uint32_t parkSeq = 0;
};

namespace {

// The kernels' view of a scene (a kernel parameter)
SceneDev scene_dev(const trq_scene* s) {
    const SceneRecords& r = s->rec;
    const PackedTree& t = s->tree;
    SceneDev d{r.spheres, r.squares, r.cubes, r.verts, r.idx, t.bvh, t.nodes, t.topSoA, t.info.topNodes, t.tris, t.sph, t.sq, t.triN, t.rootRef};
    for (int k = 0; k < 3; ++k) { d.rootMin[k] = t.rootMin[k]; d.rootMax[k] = t.rootMax[k]; }
    d.nNode = t.info.nNode;
    return d;
}

void free_scene(trq_scene* s) {
    if (!s) return;
    cudaDeviceSynchronize();                                   // launches on any stream may still read the arrays
    s->rec.release();
    s->tree.release();
    pool_free(s->d_queues);
    for (int b = 0; b < kStageBufs; ++b) {
        cudaFree(s->d_stageRays[b]); cudaFree(s->d_stageHits[b]);
        if (s->stageStream[b]) cudaStreamDestroy(s->stageStream[b]);
    }
    for (int k = 0; k < kProfRing; ++k)
        for (int j = 0; j < 3; ++j) if (s->evProf[k][j]) cudaEventDestroy(s->evProf[k][j]);
    cudaFree(s->d_profStamps);
    cudaFree(s->d_park);
    cudaFree(s->d_parkRunning);
    delete s;
}

template <typename T>
int upload(T** dst, const void* src, size_t count, cudaMemcpyKind kind) {
    *dst = nullptr;
    if (count == 0) return TRQ_OK;
    TRQ_CUDA(pool_malloc((void**)dst, count * sizeof(T)));
    TRQ_CUDA(cudaMemcpyAsync(*dst, src, count * sizeof(T), kind, nullptr));
    return TRQ_OK;
}

int upload_records(SceneRecords& r, const trq_scene_desc* d, cudaMemcpyKind kind) {
    int rc;
    if ((rc = upload(&r.spheres, d->sphereList, d->nSphere, kind)) != TRQ_OK) return rc;
    if ((rc = upload(&r.squares, d->squareList, d->nSquare, kind)) != TRQ_OK) return rc;
    if ((rc = upload(&r.cubes, d->cubeList, d->nCube, kind)) != TRQ_OK) return rc;
    if ((rc = upload(&r.verts, d->triList, d->nVert, kind)) != TRQ_OK) return rc;
    if ((rc = upload(&r.idx, d->idxList, (size_t)d->nTri * 3, kind)) != TRQ_OK) return rc;
    r.nSphere = d->nSphere; r.nSquare = d->nSquare; r.nCube = d->nCube; r.nVert = d->nVert; r.nTri = d->nTri;
    return TRQ_OK;
}

// Walk the tree once on the host: validate the layout contract and assign every reachable node its packed reference.
// Leaves are numbered per kind in depth-first order (left child first). Interior nodes: the first packed::kTopMax of a
// breadth-first walk come first, in that order (the block a kernel may stage in shared memory); the rest follow in
// depth-first order. Sets t's counts, root and maxPIndex.
int plan_layout(const trq_scene_desc* d, std::vector<uint32_t>& ref, PackedTree& t) {
    const RefBVH* N = (const RefBVH*)d->bvhList;
    const uint32_t n = d->nNode;
    ref.assign(n, TRQ_REF_DONE_WORD);
    uint32_t nTriLeaf = 0, nSphLeaf = 0, nSqLeaf = 0, nLeaf = 0, maxDepth = 0, maxPIndex = 0;
    std::vector<uint32_t> interiorDfs;                       // interior nodes in depth-first order
    struct Item { uint32_t node, depth; };
    std::vector<Item> stack;
    stack.push_back({0u, 0u});
    if (N[0].parent != 0) return trq::fail(TRQ_ERR_LAYOUT, "bvhList: the root's parent must be 0 (BVH.hh:264), found %u", N[0].parent);
    while (!stack.empty()) {
        const Item it = stack.back(); stack.pop_back();
        const uint32_t i = it.node;
        if (i >= n) return trq::fail(TRQ_ERR_LAYOUT, "bvhList: child index %u out of range (nNode %u)", i, n);
        if (ref[i] != TRQ_REF_DONE_WORD) return trq::fail(TRQ_ERR_LAYOUT, "bvhList: node %u reachable twice (not a tree)", i);
        const RefBVH& b = N[i];
        if (b.pType == TRQ_BVH) {
            if (it.depth > 31) return trq::fail(TRQ_ERR_DEPTH, "bvhList: interior depth %u exceeds the 32-bit trail (Render.hh:140)", it.depth);
            if (b.left >= n || b.right >= n)
                return trq::fail(TRQ_ERR_LAYOUT, "bvhList: child index %u out of range (nNode %u)", b.left >= n ? b.left : b.right, n);
            if (b.left == 0 || b.right == 0 || b.left == b.right)
                return trq::fail(TRQ_ERR_LAYOUT, "bvhList: interior node %u has invalid children (%u, %u)", i, b.left, b.right);
            // Scene::hit climbs through `parent` (Render.hh:153,164,197): a child that does not point back would loop
            if (N[b.left].parent != i || N[b.right].parent != i)
                return trq::fail(TRQ_ERR_LAYOUT, "bvhList: children (%u, %u) of node %u do not name it as their parent (%u, %u)",
                                 b.left, b.right, i, N[b.left].parent, N[b.right].parent);
            if (interiorDfs.size() >= 0x1fffffffu) return trq::fail(TRQ_ERR_LAYOUT, "bvhList: too many interior nodes");
            ref[i] = TRQ_MAKE_REF(REF_INTERIOR, 0);          // numbered below
            interiorDfs.push_back(i);
            maxDepth = it.depth > maxDepth ? it.depth : maxDepth;
            stack.push_back({b.right, it.depth + 1});     // left is popped (numbered) first
            stack.push_back({b.left, it.depth + 1});
        } else {
            ++nLeaf;
            if (b.pIndex > maxPIndex) maxPIndex = b.pIndex;
            switch (b.pType) {
                case TRQ_TRIANGLE:
                    if (b.pIndex >= d->nTri) return trq::fail(TRQ_ERR_LAYOUT, "leaf %u: triangle pIndex %u >= nTri %u", i, b.pIndex, d->nTri);
                    for (int k = 0; k < 3; ++k)
                        if (d->idxList[3 * (size_t)b.pIndex + k] >= d->nVert)
                            return trq::fail(TRQ_ERR_LAYOUT, "triangle %u: vertex index out of range", b.pIndex);
                    ref[i] = TRQ_MAKE_REF(REF_TRI, nTriLeaf++);
                    break;
                case TRQ_SPHERE:
                    if (b.pIndex >= d->nSphere) return trq::fail(TRQ_ERR_LAYOUT, "leaf %u: sphere pIndex %u >= nSphere %u", i, b.pIndex, d->nSphere);
                    ref[i] = TRQ_MAKE_REF(REF_SPHERE, nSphLeaf++);
                    break;
                case TRQ_SQUARE:
                    if (b.pIndex >= d->nSquare) return trq::fail(TRQ_ERR_LAYOUT, "leaf %u: square pIndex %u >= nSquare %u", i, b.pIndex, d->nSquare);
                    ref[i] = TRQ_MAKE_REF(REF_SQUARE, nSqLeaf++);
                    break;
                case TRQ_CUBE:
                    if (b.pIndex >= d->nCube) return trq::fail(TRQ_ERR_LAYOUT, "leaf %u: cube pIndex %u >= nCube %u", i, b.pIndex, d->nCube);
                    ref[i] = TRQ_MAKE_REF(REF_CUBE, i);
                    break;
                default:
                    ref[i] = TRQ_MAKE_REF(REF_NOP, i);        // Render.hh:241 `default: break`
                    break;
            }
        }
    }
    // interior numbering: breadth-first block first, then the others in depth-first order
    const uint32_t nInterior = (uint32_t)interiorDfs.size();
    uint32_t nTop = 0;
    if (nInterior) {
        std::vector<uint32_t> bfs;
        bfs.reserve(packed::kTopMax);
        bfs.push_back(0u);
        for (size_t head = 0; head < bfs.size(); ++head) {
            const RefBVH& b = N[bfs[head]];
            if (bfs.size() < packed::kTopMax && N[b.left].pType == TRQ_BVH) bfs.push_back(b.left);
            if (bfs.size() < packed::kTopMax && N[b.right].pType == TRQ_BVH) bfs.push_back(b.right);
        }
        nTop = (uint32_t)bfs.size();
        for (uint32_t k = 0; k < nTop; ++k) ref[bfs[k]] = TRQ_MAKE_REF(REF_INTERIOR, k) | 0x10000000u;   // bit 28: numbered (cleared below)
        uint32_t next = nTop;
        for (uint32_t i : interiorDfs) {
            if (ref[i] & 0x10000000u) ref[i] &= ~0x10000000u;
            else ref[i] = TRQ_MAKE_REF(REF_INTERIOR, next++);
        }
    }
    trq_scene_info_t& info = t.info;
    info.nNode = n; info.nInterior = nInterior; info.nLeaf = nLeaf; info.maxDepth = maxDepth;
    info.nTri = nTriLeaf; info.nSphere = nSphLeaf;
    info.nSquare = d->nSquare; info.nCube = d->nCube;
    info.topNodes = nTop;
    t.nSqLeaf = nSqLeaf; t.maxPIndex = maxPIndex; t.rootRef = ref[0];
    for (int k = 0; k < 3; ++k) { t.rootMin[k] = N[0].bBOX.mini[k]; t.rootMax[k] = N[0].bBOX.maxi[k]; }
    return TRQ_OK;
}

// Which launch configuration a trace uses: TRQ_CFG in the environment (experiments), else the scene's default.
int pick_cfg(const trq_scene* s) {
    static const int env = [] { const char* e = getenv("TRQ_CFG"); return e ? atoi(e) : -1; }();
    int c = (env >= 0 && env < kNumCfgs) ? env : s->defaultCfg;
    if (!s->tree.cfg[c].usable) c = 0;
    return c;
}

int launch_trace(trq_scene* s, const trq_ray* d_rays, uint64_t n, uint32_t flags, void* d_hits, cudaStream_t st,
                 const unsigned long long* nPtr = nullptr, uint32_t* tileDone = nullptr, uint32_t tileShift = 0) {
    if (n == 0) return TRQ_OK;
    const bool hit16 = (flags & TRQ_HIT16) != 0;
    const size_t recBytes = hit16 ? sizeof(trq_hit16) : sizeof(trq_hit);
    constexpr uint64_t kMaxPerLaunch = TRQ_MAX_RAYS_PER_LAUNCH;
    if (n > kMaxPerLaunch) {
        if (nPtr || tileDone) return trq::fail(TRQ_ERR_INVALID, "trq_trace_indirect / trq_trace_gather: more than 2^31 rays");
        for (uint64_t off = 0; off < n; off += kMaxPerLaunch) {
            const uint64_t m = (n - off) < kMaxPerLaunch ? (n - off) : kMaxPerLaunch;
            const int rc = launch_trace(s, d_rays + off, m, flags, (uint8_t*)d_hits + off * recBytes, st);
            if (rc != TRQ_OK) return rc;
        }
        return TRQ_OK;
    }
    const bool any = (flags & TRQ_TRACE_ANY) != 0;
    const SceneDev dev = scene_dev(s);
    // TRQ_SORT_RAYS: counting sort of ray indices by (origin cell, direction octant); stream-ordered scratch. The flag is the
    // caller's word that the batch is incoherent. Without it, scenes whose packed tree is more than twice the L2 (where an
    // incoherent batch runs at DRAM latency: C5 400 vs 990 Mrays/s) get the AUTOMATIC mode for batches of >= 1 M rays: a
    // probe over 64 K sampled rays measures how many neighbouring rays share a key, and the queue is ordered only if fewer
    // than half do -- decided on the device, no host round trip. TRQ_NO_SORT opts out; TRQ_SORT_RAYS=0/1 in the environment overrides
    // both (experiments), TRQ_AUTO_SORT=1 treats every scene as large (tests).
    static const int sortEnv = [] { const char* e = getenv("TRQ_SORT_RAYS"); return e ? atoi(e) : -1; }();
    const char* autoStr = getenv("TRQ_AUTO_SORT");               // read per call: the tests switch it inside one process
    const int autoEnv = autoStr ? atoi(autoStr) : -1;
    const bool sortRays = sortEnv >= 0 ? (sortEnv != 0) : ((flags & TRQ_SORT_RAYS) != 0);
    const bool autoSort = !sortRays && sortEnv < 0 && !(flags & TRQ_NO_SORT) && !tileDone && n >= (1ull << 20) &&
                          (autoEnv >= 0 ? autoEnv != 0 : s->tree.largeTree);
    const bool ordered = (sortRays && n >= 65536) || autoSort;
    cudaStreamCaptureStatus capture = cudaStreamCaptureStatusNone;
    TRQ_CUDA(cudaStreamIsCapturing(st, &capture));
    // Early launch (programmatic dependent launch): the packed kernel's CTAs may take the SMs that the previous kernel on
    // this stream leaves as its last, longest rays finish, instead of waiting for its last CTA (profiles/r07_pdl.txt).
    // Only for a plain eager launch of the packed kernel on a tree that has been traced as it is: not under capture (a graph
    // replay may run beside anything), not for the ordered, indirect or gather paths (their inputs are written by the kernels
    // just before them) and not right after a refit or rebuild.
    bool early = false;
#ifndef TRQ_NO_PDL
    early = !(flags & TRQ_KERNEL_REFLAYOUT) && !ordered && !nPtr && !tileDone && capture == cudaStreamCaptureStatusNone &&
            s->treeTraced.load();
#endif
    s->treeTraced.store(true);
    cudaEvent_t* prof = nullptr;
    unsigned long long* stamps = nullptr;
    if (s->profile) {
        std::lock_guard<std::mutex> lock(s->profMutex);
        if (s->profile) {
            const uint32_t slot = s->profHead % kProfRing;
            prof = s->evProf[slot];
            s->profByKernel[slot] = early;
            if (early) { stamps = s->d_profStamps + 2 * slot; prof = nullptr; }
            s->profHead++; if (s->profCount < kProfRing) s->profCount++;
        }
    }
    if (prof) TRQ_CUDA(cudaEventRecord(prof[0], st));          // the ordering pass is part of the timed traversal
    if (flags & TRQ_KERNEL_REFLAYOUT) {
        if (hit16 || tileDone) return trq::fail(TRQ_ERR_INVALID, "TRQ_KERNEL_REFLAYOUT writes trq_hit records on one device only");
        const unsigned block = 128;
        const uint64_t grid = (n + block - 1) / block;
        if (grid > 0x7fffffffull) return trq::fail(TRQ_ERR_INVALID, "trq_trace: batch too large");
        if (any) trace_reflayout_kernel<true><<<(unsigned)grid, block, 0, st>>>(dev, d_rays, (trq_hit*)d_hits, n, nPtr);
        else     trace_reflayout_kernel<false><<<(unsigned)grid, block, 0, st>>>(dev, d_rays, (trq_hit*)d_hits, n, nPtr);
        if (prof) TRQ_CUDA(cudaEventRecord(prof[1], st));
        resolve_hits_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dev, d_rays, (trq_hit*)d_hits, n, nPtr);
        g_launches += 2;
    } else {
        static const uint32_t refillMin = [] {
            const char* e = getenv("TRQ_REFILL_MIN");
            int v = e ? atoi(e) : 20;      // B200 sweeps: 16..22 within 2 % (profiles/r02_refill_sweep.txt: 20 is +1 % on C3, +2 % on C4 over 16)
            return (uint32_t)(v < 1 ? 1 : (v > 32 ? 32 : v));
        }();
        static const uint32_t leafBatch = [] {
            const char* e = getenv("TRQ_LEAF_BATCH");
            int v = e ? atoi(e) : 12;
            return (uint32_t)(v < 1 ? 1 : (v > 32 ? 32 : v));
        }();
        static const int blocksPerSMOverride =[] { const char* e = getenv("TRQ_BLOCKS_PER_SM"); return e ? atoi(e) : 0; }();
        // under trq_trace_gather the sender kernel shares every SM with this one: a one-CTA-per-SM configuration that
        // takes (nearly) all of an SM's shared memory could be locked out by a resident sender CTA that waits for it
        const int c = tileDone ? 0 : pick_cfg(s);
        const KernelCfg& K = kCfgs[c];
        const CfgState& cs = s->tree.cfg[c];
        int perSM = cs.blocksPerSM[any ? 1 : 0][hit16 ? 1 : 0];                  // queried once, in trq_scene_create
        if (blocksPerSMOverride > 0 && blocksPerSMOverride < perSM) perSM = blocksPerSMOverride;
        uint64_t grid = (uint64_t)perSM * (uint64_t)s->numSMs;             // persistent: a multiple of the SM count
        const uint64_t need = (n + K.block - 1) / K.block;
        if (grid > need) grid = need;
        TraceParams P{};
        P.rays = d_rays; P.hits = d_hits; P.n = n;
        // Work-queue head. An eager launch takes the next one of the ring (zero: heads are zeroed at creation and every launch's
        // last CTA re-arms the one it used). A launch captured into a CUDA graph is fixed in the graph and may be replayed at
        // any later time, beside any other launch: it gets a head of its own, allocated, zeroed and freed in stream order
        // around the kernel at every replay. (A per-launch memset for eager launches too costs ~1 % on C1 / C2.)
        QueueHead* ownHead = nullptr;
        if (capture != cudaStreamCaptureStatusNone) {
            TRQ_CUDA(cudaMallocFromPoolAsync((void**)&ownHead, sizeof(QueueHead), s->scratchPool, st));
            TRQ_CUDA(cudaMemsetAsync(ownHead, 0, sizeof(QueueHead), st));
        }
        P.queue = ownHead ? ownHead : s->d_queues + (s->queueNext.fetch_add(1) % kQueueRing);
        P.stackDepth = cs.stackDepth; P.refillMin = refillMin; P.leafBatch = leafBatch;
        P.topCount = K.top ? cs.topCount : 0;
        P.order = nullptr; P.nPtr = nPtr;
        P.tileDone = tileDone; P.tileShift = tileShift;
        P.early = early ? 1u : 0u; P.timing = stamps;
#ifdef TRQ_TAIL_TIMELINE
        P.tailSlot = s->tailSeq++;
#endif
        uint32_t* scratch = nullptr;
        if (ordered) {
            const size_t words = (size_t)TRQ_SORT_BINS + 4 + 2 * (size_t)n;      // hist | ctrl | keys | order
            TRQ_CUDA(cudaMallocFromPoolAsync((void**)&scratch, words * sizeof(uint32_t), s->scratchPool, st));
            uint32_t* hist = scratch; uint32_t* ctrl = scratch + TRQ_SORT_BINS; uint32_t* keys = ctrl + 4; uint32_t* order = keys + n;
            TRQ_CUDA(cudaMemsetAsync(hist, 0, ((size_t)TRQ_SORT_BINS + 4) * sizeof(uint32_t), st));
            unsigned gb = (unsigned)((n + 255) / 256);
            if (gb > (unsigned)s->numSMs * 32u) gb = (unsigned)s->numSMs * 32u;   // grid-stride beyond that
            uint32_t* decide = autoSort ? ctrl : nullptr;
            if (autoSort) { sort_probe_kernel<<<256, 256, 0, st>>>(dev, d_rays, n, nPtr, ctrl); g_launches++; }
            sort_count_kernel<<<gb, 256, 0, st>>>(dev, d_rays, n, nPtr, keys, hist, decide);
            sort_scan_kernel<<<1, 1024, 0, st>>>(hist, decide);
            sort_scatter_kernel<<<gb, 256, 0, st>>>(keys, n, nPtr, hist, order, decide);
            g_launches += 3;
            P.order = order;
            P.orderFlag = decide;
        }
        void* args[2] = {(void*)&dev, (void*)&P};
        const void* fn = K.fn[s->tree.leaves][any ? 1 : 0][hit16 ? 1 : 0];
        std::unique_lock<std::mutex> parkLock;                  // held until the launch: halves alternate in stream order
        if (early) {
            parkLock = std::unique_lock<std::mutex>(s->parkMutex);
            if (!s->parkBound && cudaMalloc((void**)&s->d_parkRunning, 2 * sizeof(uint32_t)) == cudaSuccess &&
                cudaMemset(s->d_parkRunning, 0, 2 * sizeof(uint32_t)) == cudaSuccess) {
                s->parkStream = st; s->parkBound = true;
            }
            cudaGetLastError();
            const size_t half = (size_t)grid * (K.block / 32) * TRQ_PARK_ROWS * 128u * sizeof(float4);
            if (s->parkBound && s->parkStream == st && half > s->parkHalf) {
                if (s->d_park) {                                // the launches that use the old halves are on this stream
                    TRQ_CUDA(cudaStreamSynchronize(st));
                    TRQ_CUDA(cudaFree(s->d_park));
                    s->d_park = nullptr; s->parkHalf = 0;
                }
                if (cudaMalloc((void**)&s->d_park, 2 * half) == cudaSuccess) s->parkHalf = half;
                else { cudaGetLastError(); s->d_park = nullptr; }   // without scratch the warps wait after their first rays
            }
            if (s->parkBound && s->parkStream == st && s->d_park) {
                const uint32_t h = s->parkSeq++ & 1u;
                P.park = reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(s->d_park) + h * s->parkHalf);
                P.parkRunning = s->d_parkRunning + h;
                P.prevRunning = s->d_parkRunning + (h ^ 1u);
            }
        }
        if (early) {
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attr[0].val.programmaticStreamSerializationAllowed = 1;
            cudaLaunchConfig_t lc = {};
            lc.gridDim = dim3((unsigned)grid); lc.blockDim = dim3((unsigned)K.block); lc.dynamicSmemBytes = cs.smem; lc.stream = st;
            lc.attrs = attr; lc.numAttrs = 1;
            TRQ_CUDA(cudaLaunchKernelExC(&lc, fn, args));
        } else {
            TRQ_CUDA(cudaLaunchKernel(fn, dim3((unsigned)grid), dim3((unsigned)K.block), args, cs.smem, st));
        }
        g_launches++;
        if (ownHead) TRQ_CUDA(cudaFreeAsync(ownHead, st));
        if (scratch) TRQ_CUDA(cudaFreeAsync(scratch, st));
        if (prof) TRQ_CUDA(cudaEventRecord(prof[1], st));
    }
    if (prof) TRQ_CUDA(cudaEventRecord(prof[2], st));
    TRQ_CUDA(cudaGetLastError());
    return TRQ_OK;
}

#ifdef TRQ_STAGE_TIMELINE
// developer instrumentation (make EXTRA=-DTRQ_STAGE_TIMELINE): device timestamps around every staged operation
std::vector<cudaEvent_t> g_tl;
cudaEvent_t* timeline_events(int k) {
    const size_t at = g_tl.size();
    g_tl.resize(at + k);
    for (int i = 0; i < k; ++i) cudaEventCreate(&g_tl[at + i]);
    return &g_tl[at];
}
void timeline_dump() {
    if (getenv("TRQ_STAGE_TIMELINE_PRINT"))
        for (size_t i = 0; i + 3 < g_tl.size(); i += 4) {
            float a, b, c, d;
            cudaEventElapsedTime(&a, g_tl[0], g_tl[i]); cudaEventElapsedTime(&b, g_tl[0], g_tl[i + 1]);
            cudaEventElapsedTime(&c, g_tl[0], g_tl[i + 2]); cudaEventElapsedTime(&d, g_tl[0], g_tl[i + 3]);
            fprintf(stderr, "chunk %3zu  h2d %8.1f..%8.1f  trace ..%8.1f  d2h ..%8.1f us\n", i / 4, a * 1e3, b * 1e3, c * 1e3, d * 1e3);
        }
    for (cudaEvent_t e : g_tl) cudaEventDestroy(e);
    g_tl.clear();
}
#endif

int sync_staging(trq_scene* s) {
    for (int b = 0; b < kStageBufs; ++b)
        if (s->stageStream[b]) TRQ_CUDA(cudaStreamSynchronize(s->stageStream[b]));
    return TRQ_OK;
}

int ensure_staging(trq_scene* s, uint64_t chunk) {
    if (!s->stageReady) {
        for (int b = 0; b < kStageBufs; ++b) TRQ_CUDA(cudaStreamCreateWithFlags(&s->stageStream[b], cudaStreamNonBlocking));
        s->stageReady = true;
    }
    if (chunk > s->stageCap) {
        int rc = sync_staging(s);                             // asynchronous calls may still be using the old buffers
        if (rc != TRQ_OK) return rc;
        for (int b = 0; b < kStageBufs; ++b) {
            cudaFree(s->d_stageRays[b]); cudaFree(s->d_stageHits[b]);
            s->d_stageRays[b] = nullptr; s->d_stageHits[b] = nullptr;
        }
        s->stageCap = 0;
        for (int b = 0; b < kStageBufs; ++b) {
            TRQ_CUDA(cudaMalloc((void**)&s->d_stageRays[b], chunk * sizeof(trq_ray)));
            TRQ_CUDA(cudaMalloc((void**)&s->d_stageHits[b], chunk * sizeof(trq_hit)));
        }
        s->stageCap = chunk;
    }
    return TRQ_OK;
}

// Host-pointer path: the batch is cut into chunks; chunk k goes through staging buffer k % kStageBufs on that
// buffer's own stream (copy in, trace, copy out, in stream order). Different chunks overlap on the two copy engines
// and the SMs, buffer reuse is ordered by the stream itself, and a chunk costs four driver calls.
// Measured alternatives that did not beat it on B200 (profiles/r02_e2e_staging_experiment.txt): all H2D copies on one
// dedicated stream and all D2H copies on another, chained to the kernels by events (-4 %); chunk sizes ramping up at the
// front and down at the back of a synchronous call (no change). With a 16-byte record (TRQ_HIT16) the D2H side halves.
int trace_host(trq_scene* s, const trq_ray* rays, uint64_t n, uint32_t flags, void* hits) {
    const uint64_t chunkRays = [] {                           // read per call so that one process can sweep it
        const char* e = getenv("TRQ_CHUNK_RAYS");
        long long v = e ? atoll(e) : (TRQ_DEFAULT_CHUNK_RAYS)  /* B200 sweep: profiles/r01_e2e_chunk_sweep.txt */;
        return (uint64_t)(v < 1024 ? 1024 : v);
    }();
    const size_t recBytes = (flags & TRQ_HIT16) ? sizeof(trq_hit16) : sizeof(trq_hit);
    std::lock_guard<std::mutex> lock(s->stageMutex);
    // a sorted chunk is only as coherent as it is large: C5 e2e 461 / 605 / 599 / 504 Mrays/s at 512K / 1M / 2M / 4M rays
    // (the same chunk size for a tree much larger than L2 without the hint: the automatic mode looks at batches of >= 2^20 rays)
    const bool mayOrder = (flags & TRQ_SORT_RAYS) || (s->tree.largeTree && !(flags & TRQ_NO_SORT));
    const uint64_t want = mayOrder ? 2 * chunkRays : chunkRays;
    const uint64_t chunk = n < want ? n : want;
    int rc = ensure_staging(s, chunk);
    if (rc != TRQ_OK) return rc;
    uint64_t done = 0;
    while (done < n) {
        const uint64_t m = (n - done) < chunk ? (n - done) : chunk;
        const int b = (int)(s->stageSeq++ % kStageBufs);       // runs across calls: TRQ_HOST_ASYNC calls share the ring
        cudaStream_t st = s->stageStream[b];
#ifdef TRQ_STAGE_TIMELINE
        cudaEvent_t* tl = timeline_events(4); cudaEventRecord(tl[0], st);
#endif
        TRQ_CUDA(cudaMemcpyAsync(s->d_stageRays[b], rays + done, m * sizeof(trq_ray), cudaMemcpyHostToDevice, st));
#ifdef TRQ_STAGE_TIMELINE
        cudaEventRecord(tl[1], st);
#endif
        rc = launch_trace(s, s->d_stageRays[b], m, flags, s->d_stageHits[b], st);
        if (rc != TRQ_OK) return rc;
#ifdef TRQ_STAGE_TIMELINE
        cudaEventRecord(tl[2], st);
#endif
        TRQ_CUDA(cudaMemcpyAsync((uint8_t*)hits + done * recBytes, s->d_stageHits[b], m * recBytes, cudaMemcpyDeviceToHost, st));
#ifdef TRQ_STAGE_TIMELINE
        cudaEventRecord(tl[3], st);
#endif
        done += m;
    }
#ifdef TRQ_STAGE_TIMELINE
    sync_staging(s); timeline_dump();
#endif
    if (flags & TRQ_HOST_ASYNC) return TRQ_OK;               // the caller collects with trq_host_sync()
    return sync_staging(s);
}

}  // namespace

extern "C" {

int trq_version(void) { return TRQ_VERSION; }

const char* trq_last_error_string(void) { return trq::last_error(); }

int trq_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

uint64_t trq_launch_count(void) { return g_launches.load(); }

#ifdef TRQ_TAIL_TIMELINE
// tools/tail_probe.py: out <- the stamps of the last TRQ_TAIL_LAUNCHES packed-kernel launches ([launch % 8][CTA][start,
// ~first exhausted, exit]); reset: clear them and number this scene's launches from 0 again
int trq_debug_tail(trq_scene* s, unsigned long long* out, int reset) {
    TRQ_CUDA(cudaDeviceSynchronize());
    if (out) TRQ_CUDA(cudaMemcpyFromSymbol(out, trq::g_tail, sizeof(trq::g_tail)));
    if (reset) {
        void* p = nullptr;
        TRQ_CUDA(cudaGetSymbolAddress(&p, trq::g_tail));
        TRQ_CUDA(cudaMemset(p, 0, sizeof(trq::g_tail)));
        TRQ_CUDA(cudaDeviceSynchronize());
        s->tailSeq = 0;
    }
    return TRQ_OK;
}
#endif

#ifdef TRQ_STATS
void trq_debug_stats(unsigned long long* out, int reset) {
    cudaMemcpyFromSymbol(out, trq::g_stats, sizeof(unsigned long long) * 8);
    if (reset) { unsigned long long z[8] = {0}; cudaMemcpyToSymbol(trq::g_stats, z, sizeof z); }
}
#endif

}  // extern "C"

namespace {

int check_desc(const trq_scene_desc* d, trq_scene** out, const char* who) {
    if (!d || !out) return trq::fail(TRQ_ERR_INVALID, "%s: NULL argument", who);
    *out = nullptr;
    if (!d->bvhList || d->nNode == 0) return trq::fail(TRQ_ERR_INVALID, "%s: empty bvhList", who);
    if ((d->nSphere && !d->sphereList) || (d->nSquare && !d->squareList) || (d->nCube && !d->cubeList) ||
        (d->nVert && !d->triList) || (d->nTri && !d->idxList))
        return trq::fail(TRQ_ERR_INVALID, "%s: NULL array with non-zero count", who);
    return TRQ_OK;
}

// Launch configurations for the tree (t.stackDepth, t.leaves set): per-CTA shared memory = staged top-of-tree nodes +
// far-child stack + cold per-ray words, resident CTAs per SM, usability; and the automatic choice t.autoCfg.
int size_configs(PackedTree& t) {
    for (int c = 0; c < kNumCfgs; ++c) {
        const KernelCfg& K = kCfgs[c];
        CfgState& cs = t.cfg[c];
        cs.stackDepth = t.stackDepth;
        const size_t perRay = ((size_t)cs.stackDepth + COLD_WORDS) * K.block * sizeof(uint32_t);
        size_t budget = kSmemPerSM / (size_t)K.minb - kSmemBlockReserve;
        if (budget > kSmemDynamicMax) budget = kSmemDynamicMax;
        cs.topCount = 0;
        if (K.top) {
            const char* topStr = getenv("TRQ_TOP_NODES");               // read per scene: the sweeps create one scene per value
            const int topEnv = topStr ? atoi(topStr) : -1;
            if (budget > perRay) cs.topCount = (uint32_t)((budget - perRay) / packed::kNodeBytes);
            if (cs.topCount > t.info.topNodes) cs.topCount = t.info.topNodes;
            if (topEnv >= 0 && (uint32_t)topEnv < cs.topCount) cs.topCount = (uint32_t)topEnv;
        }
        cs.smem = perRay + (size_t)cs.topCount * packed::kNodeBytes;
        cs.usable = cs.smem <= kSmemDynamicMax && !(K.top && cs.topCount == 0 && c != 0);
        if (!cs.usable) continue;
        cudaError_t e = cudaSuccess;
        for (int a = 0; a < 2 && e == cudaSuccess; ++a)
            for (int f = 0; f < 2 && e == cudaSuccess; ++f) {
                const void* fn = K.fn[t.leaves][a][f];
                if (cs.smem > 48 * 1024) e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemDynamicMax);
                if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cs.blocksPerSM[a][f], fn, K.block, cs.smem);
                if (e == cudaSuccess && cs.blocksPerSM[a][f] < 1) cs.usable = false;
            }
        if (e != cudaSuccess) {
            if (c == 0) return trq::fail(TRQ_ERR_CUDA, "trace_packed_kernel (%s) occupancy query failed: %s", K.name, cudaGetErrorString(e));
            cudaGetLastError();                                // an optional configuration that does not fit: not offered
            cs.usable = false;
        }
    }
    if (!t.cfg[0].usable) return trq::fail(TRQ_ERR_CUDA, "trace_packed_kernel does not fit on an SM (smem %zu)", t.cfg[0].smem);
    // Staging pays when the staged block IS the tree (C1: +2-15 %); with the leaf-specialised kernels it no longer does when
    // only the top levels fit (C2 / the reference's Cornell mix: -3 to -6 %), and it loses clearly on 1 M+ triangle scenes
    // (profiles/r02_top_of_tree_experiment.txt): chosen only for trees that fit whole.
    t.autoCfg = 0;
    for (int c = 1; c < kNumCfgs; ++c)
        if (kCfgs[c].top && t.cfg[c].usable && t.info.nInterior <= t.cfg[c].topCount) { t.autoCfg = c; break; }
    return TRQ_OK;
}

// Derives t's packed arrays from its nodes and the records, on the device (creation and refit).
void launch_pack(const PackedTree& t, const SceneRecords& r) {
    const unsigned block = 256, grid = (t.info.nNode + block - 1) / block;
    pack_scene_kernel<<<grid, block>>>(t.bvh, t.ref, t.info.nNode, r.verts, r.idx, r.spheres, r.squares,
                                       t.nodes, t.tris, t.sph, t.sq, t.triN, t.topSoA, t.info.topNodes);
    g_launches++;
}

// The part of building a tree that is the same for every path: t.bvh and t.ref are resident, t's counts, root and maxPIndex
// are set (plan_layout or plan_tree). Allocates the packed arrays, derives them on the device and sizes the launch
// configurations.
int pack_tree(PackedTree& t, const SceneRecords& r, int device) {
    StageTimer tm;
    trq_scene_info_t& info = t.info;
    const packed::Sizes b = packed::sizes(info.nInterior, info.nTri, info.nSphere, t.nSqLeaf, info.topNodes);
    if (b.nodes && pool_malloc((void**)&t.nodes, b.nodes) != cudaSuccess) return trq::fail(TRQ_ERR_CUDA, "cudaMalloc(nodes %zu B) failed", b.nodes);
    if (b.tris && pool_malloc((void**)&t.tris, b.tris) != cudaSuccess) return trq::fail(TRQ_ERR_CUDA, "cudaMalloc(tris %zu B) failed", b.tris);
    if (b.sph && pool_malloc((void**)&t.sph, b.sph) != cudaSuccess) return trq::fail(TRQ_ERR_CUDA, "cudaMalloc(spheres %zu B) failed", b.sph);
    if (b.sq && pool_malloc((void**)&t.sq, b.sq) != cudaSuccess) return trq::fail(TRQ_ERR_CUDA, "cudaMalloc(squares %zu B) failed", b.sq);
    if (b.triN && pool_malloc((void**)&t.triN, b.triN) != cudaSuccess) return trq::fail(TRQ_ERR_CUDA, "cudaMalloc(triangle normals %zu B) failed", b.triN);
    if (b.top && pool_malloc((void**)&t.topSoA, b.top) != cudaSuccess) return trq::fail(TRQ_ERR_CUDA, "cudaMalloc(top-of-tree block) failed");
    TRQ_LAP(tm, "allocate packed arrays");
    launch_pack(t, r);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return trq::fail(TRQ_ERR_CUDA, "pack_scene_kernel failed: %s", cudaGetErrorString(e));
    TRQ_LAP(tm, "pack_scene_kernel");
    t.stackDepth = info.maxDepth + 1;
    // (a leaf of unknown pType, which dispatches to `default: break`, also selects the general kernels)
    t.leaves = info.nLeaf == info.nTri ? LEAVES_TRI : (info.nLeaf == info.nTri + info.nSphere ? LEAVES_TRI_SPHERE : LEAVES_ALL);
    int rc = size_configs(t);
    if (rc != TRQ_OK) return rc;
    TRQ_LAP(tm, "kernel configurations");

    info.bytesReferenceLayout = (uint64_t)r.nSphere * sizeof(RefSphere) + (uint64_t)r.nSquare * sizeof(RefSquare) +
                                (uint64_t)r.nCube * sizeof(RefCube) + (uint64_t)r.nVert * sizeof(RefVertex) +
                                (uint64_t)r.nTri * 12 + (uint64_t)info.nNode * sizeof(RefBVH);
    info.bytesPacked = b.nodes + b.tris + b.sph + b.sq + b.triN;
    {
        int l2 = 0;
        if (cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, device) != cudaSuccess) { cudaGetLastError(); l2 = 0; }
        t.largeTree = l2 > 0 && (uint64_t)(b.nodes + b.tris + b.sph + b.sq) > 2ull * (uint64_t)l2;   // what traversal touches
    }
    info.device = device;
    return TRQ_OK;
}

int open_scene(int device, trq_scene** sOut, const char* who) {
    int ndev = trq_device_count();
    if (ndev <= 0) return trq::fail(TRQ_ERR_NO_DEVICE, "%s: no CUDA device (there is no CPU fallback)", who);
    if (device < 0 || device >= ndev) return trq::fail(TRQ_ERR_INVALID, "%s: device %d out of range (%d devices)", who, device, ndev);
    trq_scene* s = new (std::nothrow) trq_scene();
    if (!s) return trq::fail(TRQ_ERR_NOMEM, "%s: out of host memory", who);
    s->device = device;
    if (cudaDeviceGetAttribute(&s->numSMs, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) { delete s; return trq::fail(TRQ_ERR_CUDA, "cudaDeviceGetAttribute failed"); }
    *sOut = s;
    return TRQ_OK;
}

// What a scene keeps whatever its tree: the zeroed ray-queue heads of eager launches and the TRQ_SORT_RAYS scratch pool
// (stream-ordered, kept between launches). Runs on the scene's device before the creation's first synchronisation.
int open_queues(trq_scene* s) {
    if (pool_malloc((void**)&s->d_queues, kQueueRing * sizeof(QueueHead)) != cudaSuccess) return trq::fail(TRQ_ERR_CUDA, "cudaMalloc(queue heads) failed");
    if (cudaMemsetAsync(s->d_queues, 0, kQueueRing * sizeof(QueueHead), nullptr) != cudaSuccess) return trq::fail(TRQ_ERR_CUDA, "cudaMemset(queue heads) failed");
    s->scratchPool = trq::scratch_pool(s->device);
    if (!s->scratchPool) return trq::fail(TRQ_ERR_CUDA, "cudaMemPoolCreate failed");
    return TRQ_OK;
}

const char* plan_error_text(uint32_t code) {
    switch (code) {
        case plan::ERR_CHILD_RANGE: return "child index out of range";
        case plan::ERR_CHILDREN:    return "interior node has invalid children";
        case plan::ERR_PARENT_LINK: return "parent / child links do not agree (not a tree)";
        case plan::ERR_ROOT_PARENT: return "the root's parent must be 0 (BVH.hh:264)";
        case plan::ERR_LEAF_INDEX:  return "leaf pIndex out of range";
        case plan::ERR_VERTEX_INDEX: return "triangle vertex index out of range";
        case plan::ERR_DEPTH:       return "interior depth exceeds the 32-bit trail (Render.hh:140)";
        case plan::ERR_UNREACHABLE: return "nodes not reachable from the root";
        default: return "unknown";
    }
}

// Device planning, shared by trq_scene_create_device and trq_scene_rebuild: t.bvh (nNode nodes over the records r) is
// resident. The planning kernels (kernels/plan_scene.cuh) validate the tree and number it into a new t.ref, and 128 bytes of
// counters come back with t's counts, root and maxPIndex.
int plan_tree(PackedTree& t, uint32_t n, const SceneRecords& r, int device, const char* who) {
    StageTimer tm;
    if (pool_malloc((void**)&t.ref, (size_t)n * sizeof(uint32_t)) != cudaSuccess) return trq::fail(TRQ_ERR_CUDA, "%s: cudaMalloc(refs) failed", who);
    plan::PlanInfo hostInfo;
    {
        trq::PoolScratch mem(device, nullptr);
        plan::Counts* cnt; uint32_t *leafTotal, *arrivals, *pre, *topPos, *sortedPre; plan::PlanInfo* dInfo;
        if (!(mem.alloc(&cnt, n) && mem.alloc(&leafTotal, n) && mem.alloc(&arrivals, n) && mem.alloc(&pre, n) && mem.alloc(&topPos, n) &&
              mem.alloc(&sortedPre, 2048) && mem.alloc(&dInfo, 1)))
            return trq::fail(TRQ_ERR_NOMEM, "%s: out of device memory", who);
        cudaMemsetAsync(arrivals, 0, (size_t)n * 4); cudaMemsetAsync(topPos, 0, (size_t)n * 4);
        cudaMemsetAsync(cnt, 0, (size_t)n * sizeof(plan::Counts)); cudaMemsetAsync(leafTotal, 0, (size_t)n * 4);
        cudaMemsetAsync(dInfo, 0, sizeof(plan::PlanInfo)); cudaMemsetAsync(t.ref, 0xff, (size_t)n * 4);
        const unsigned grid = (n + 255) / 256;
        plan::validate_kernel<<<grid, 256>>>(t.bvh, n, r.nSphere, r.nSquare, r.nCube, r.nTri, r.nVert, r.idx, dInfo);
        plan::counts_kernel<<<grid, 256>>>(t.bvh, n, cnt, leafTotal, arrivals);
        plan::number_kernel<<<grid, 256>>>(t.bvh, n, cnt, leafTotal, t.ref, pre, dInfo);
        plan::top_block_kernel<<<1, 1024>>>(t.bvh, n, pre, topPos, sortedPre, dInfo);
        plan::refs_kernel<<<grid, 256>>>(t.bvh, n, pre, topPos, sortedPre, t.ref, dInfo);
        g_launches += 5;
        cudaError_t e = cudaMemcpy(&hostInfo, dInfo, sizeof hostInfo, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) return trq::fail(TRQ_ERR_CUDA, "%s: planning kernels failed: %s", who, cudaGetErrorString(e));
    }
    TRQ_LAP(tm, "plan kernels");
    if (hostInfo.error)
        return trq::fail(hostInfo.error == plan::ERR_DEPTH ? TRQ_ERR_DEPTH : TRQ_ERR_LAYOUT, "bvhList: node %u: %s (%u, %u)", hostInfo.errorNode,
                         plan_error_text(hostInfo.error), hostInfo.errorA, hostInfo.errorB);
    trq_scene_info_t& info = t.info;
    info.nNode = n; info.nInterior = hostInfo.nInterior; info.nLeaf = hostInfo.nLeaf; info.maxDepth = hostInfo.maxDepth;
    info.nTri = hostInfo.nTri; info.nSphere = hostInfo.nSphere; info.nSquare = r.nSquare; info.nCube = r.nCube;
    info.topNodes = hostInfo.nTop;
    t.nSqLeaf = hostInfo.nSquare; t.maxPIndex = hostInfo.maxPIndex; t.rootRef = hostInfo.rootRef;
    for (int k = 0; k < 3; ++k) { t.rootMin[k] = hostInfo.rootMin[k]; t.rootMax[k] = hostInfo.rootMax[k]; }
    return TRQ_OK;
}

// The refit of trq_scene_update_vertices and trq_scene_update_primitives (header: what changes and what is kept). `c` is
// checked: each list that is non-NULL with a non-zero count replaces the scene's records of that kind whole (host pointers
// with TRQ_HOST_PTRS, device pointers otherwise); idxList / bvhList are not read. Scratch is allocated before the first
// copy, so running out of memory leaves the scene as it was. The leaf kernels of the replaced kinds run, then the interior
// nodes bottom-up as unions of their children (BVH.hh:229-231), then the packed layout is derived again; all on the device.
int refit_scene(trq_scene* s, const trq_scene_desc* c, uint32_t flags, const char* who) {
    DeviceGuard guard(s->device);
    if (!guard.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", s->device);
    TRQ_CUDA(cudaDeviceSynchronize());                           // traces in flight still read the old boxes and records
    s->treeTraced.store(false);                                  // the next trace reads the new tree: no early launch
    PackedTree& t = s->tree;
    const SceneRecords& r = s->rec;
    const uint32_t n = t.info.nNode;
    trq::PoolScratch mem(s->device, nullptr);
    uint32_t* arrivals;
    if (!mem.alloc(&arrivals, n)) return trq::fail(TRQ_ERR_NOMEM, "%s: out of device memory", who);
    const cudaMemcpyKind kind = (flags & TRQ_HOST_PTRS) ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    const bool sph = c->sphereList && c->nSphere, sq = c->squareList && c->nSquare, cube = c->cubeList && c->nCube, tri = c->triList && c->nVert;
    if (sph) TRQ_CUDA(cudaMemcpy(r.spheres, c->sphereList, (size_t)c->nSphere * sizeof(RefSphere), kind));
    if (sq) TRQ_CUDA(cudaMemcpy(r.squares, c->squareList, (size_t)c->nSquare * sizeof(RefSquare), kind));
    if (cube) TRQ_CUDA(cudaMemcpy(r.cubes, c->cubeList, (size_t)c->nCube * sizeof(RefCube), kind));
    if (tri) TRQ_CUDA(cudaMemcpy(r.verts, c->triList, (size_t)c->nVert * sizeof(RefVertex), kind));
    TRQ_CUDA(cudaMemsetAsync(arrivals, 0, (size_t)n * 4));
    const unsigned grid = (n + 255) / 256;
    if (tri) { plan::refit_leaves_kernel<<<grid, 256>>>(t.bvh, t.ref, n, r.verts, r.idx); g_launches++; }
    if (sph || sq || cube) {
        const int rc = trq::refit_primitive_leaves_on_device(t.bvh, t.ref, n, sph ? r.spheres : nullptr, sq ? r.squares : nullptr,
                                                             cube ? r.cubes : nullptr);
        if (rc != TRQ_OK) return rc;
    }
    plan::refit_interior_kernel<<<grid, 256>>>(t.bvh, t.ref, n, arrivals);
    g_launches++;
    launch_pack(t, r);
    RefAABB root;
    TRQ_CUDA(cudaMemcpy(&root, &t.bvh[0].bBOX, sizeof root, cudaMemcpyDeviceToHost));
    for (int k = 0; k < 3; ++k) { t.rootMin[k] = root.mini[k]; t.rootMax[k] = root.maxi[k]; }
    TRQ_CUDA(cudaGetLastError());
    return TRQ_OK;
}

}  // namespace

extern "C" {

int trq_scene_create(const trq_scene_desc* d, int device, trq_scene** out) {
    int rc = check_desc(d, out, "trq_scene_create");
    if (rc != TRQ_OK) return rc;

    PackedTree tree;
    std::vector<uint32_t> ref;
    rc = plan_layout(d, ref, tree);                            // pure host validation: runs without a GPU
    if (rc != TRQ_OK) return rc;

    trq_scene* s = nullptr;
    if ((rc = open_scene(device, &s, "trq_scene_create")) != TRQ_OK) return rc;
    s->tree = tree;
    DeviceGuard guard(device);
    auto bail = [&](int code) { free_scene(s); return code; };
    if (!guard.ok) return bail(trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", device));
    const cudaMemcpyKind k = cudaMemcpyHostToDevice;
    if ((rc = open_queues(s)) != TRQ_OK) return bail(rc);
    if ((rc = upload_records(s->rec, d, k)) != TRQ_OK) return bail(rc);
    if ((rc = upload(&s->tree.bvh, d->bvhList, d->nNode, k)) != TRQ_OK) return bail(rc);
    if ((rc = upload(&s->tree.ref, ref.data(), ref.size(), k)) != TRQ_OK) return bail(rc);
    if ((rc = pack_tree(s->tree, s->rec, device)) != TRQ_OK) return bail(rc);
    s->defaultCfg = s->tree.autoCfg;
    *out = s;
    return TRQ_OK;
}

// Device-resident input: the six arrays are DEVICE pointers on `device` (e.g. the node array trq_bvh_build_tree_device
// just produced). They are copied device to device, and validation + numbering run as kernels (kernels/plan_scene.cuh):
// no array crosses PCIe, 128 bytes of counters come back.
int trq_scene_create_device(const trq_scene_desc* d, int device, trq_scene** out) {
    int rc = check_desc(d, out, "trq_scene_create_device");
    if (rc != TRQ_OK) return rc;
    trq_scene* s = nullptr;
    if ((rc = open_scene(device, &s, "trq_scene_create_device")) != TRQ_OK) return rc;
    DeviceGuard guard(device);
    auto bail = [&](int code) { free_scene(s); return code; };
    if (!guard.ok) return bail(trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", device));
    StageTimer tm;
    TRQ_LAP(tm, "open scene");
    const cudaMemcpyKind k = cudaMemcpyDeviceToDevice;
    if ((rc = open_queues(s)) != TRQ_OK) return bail(rc);
    if ((rc = upload_records(s->rec, d, k)) != TRQ_OK) return bail(rc);
    if ((rc = upload(&s->tree.bvh, d->bvhList, d->nNode, k)) != TRQ_OK) return bail(rc);
    TRQ_LAP(tm, "copy six arrays D2D");
    if ((rc = plan_tree(s->tree, d->nNode, s->rec, device, "trq_scene_create_device")) != TRQ_OK) return bail(rc);
    if ((rc = pack_tree(s->tree, s->rec, device)) != TRQ_OK) return bail(rc);
    s->defaultCfg = s->tree.autoCfg;
    *out = s;
    return TRQ_OK;
}

// Refit after the vertices moved (animated meshes): the refit with only triList replaced.
int trq_scene_update_vertices(trq_scene* s, const void* triList, uint32_t nVert, uint32_t flags) {
    if (!s || !triList) return trq::fail(TRQ_ERR_INVALID, "trq_scene_update_vertices: NULL argument");
    if (nVert != s->rec.nVert) return trq::fail(TRQ_ERR_INVALID, "trq_scene_update_vertices: %u vertices, the scene has %u", nVert, s->rec.nVert);
    if (nVert == 0) return TRQ_OK;                              // (a one-leaf scene is refit too: its leaf is the root)
    trq_scene_desc c{};
    c.triList = triList; c.nVert = nVert;
    return refit_scene(s, &c, flags, "trq_scene_update_vertices");
}

// Refit after spheres, squares, cubes and / or vertices moved: every check comes before the scene is touched.
int trq_scene_update_primitives(trq_scene* s, const trq_scene_desc* c, uint32_t flags) {
    const char* who = "trq_scene_update_primitives";
    if (!s || !c) return trq::fail(TRQ_ERR_INVALID, "%s: NULL argument", who);
    if (c->idxList || c->nTri || c->bvhList || c->nNode)
        return trq::fail(TRQ_ERR_INVALID, "%s: idxList and bvhList must be NULL with count 0 (they would change the topology)", who);
    if ((c->nSphere && !c->sphereList) || (c->nSquare && !c->squareList) || (c->nCube && !c->cubeList) || (c->nVert && !c->triList))
        return trq::fail(TRQ_ERR_INVALID, "%s: NULL array with non-zero count", who);
    const struct { const void* list; uint32_t n, have; const char* what; } kinds[] = {
        {c->sphereList, c->nSphere, s->rec.nSphere, "spheres"}, {c->squareList, c->nSquare, s->rec.nSquare, "squares"},
        {c->cubeList, c->nCube, s->rec.nCube, "cubes"}, {c->triList, c->nVert, s->rec.nVert, "vertices"}};
    for (const auto& k : kinds)
        if (k.list && k.n != k.have) return trq::fail(TRQ_ERR_INVALID, "%s: %u %s, the scene has %u", who, k.n, k.what, k.have);
    return refit_scene(s, c, flags, who);
}

// New topology from the current geometry (header: the leaf list, the records and what a rebuild keeps). A new tree is built
// over the scene's records (with the new vertices, when given), planned and packed like trq_scene_create_device's; only then
// is it swapped into the scene and the old tree released, so a failure leaves the scene as it was.
int trq_scene_rebuild(trq_scene* s, const void* triList, uint32_t nVert, uint32_t flags) {
    if (!s) return trq::fail(TRQ_ERR_INVALID, "trq_scene_rebuild: NULL scene");
    if (triList ? nVert != s->rec.nVert : (nVert != 0 && nVert != s->rec.nVert))
        return trq::fail(TRQ_ERR_INVALID, "trq_scene_rebuild: %u vertices, the scene has %u", nVert, s->rec.nVert);
    DeviceGuard guard(s->device);
    if (!guard.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", s->device);
    TRQ_CUDA(cudaDeviceSynchronize());                           // traces in flight still read the old arrays
    PackedTree t;
    RefVertex* newVerts = nullptr;                               // owned here until the commit
    auto bail = [&](int code) { t.release(); pool_free(newVerts); return code; };
    int rc = TRQ_OK;
    if (triList && nVert && (rc = upload(&newVerts, triList, nVert, (flags & TRQ_HOST_PTRS) ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice)) != TRQ_OK)
        return bail(rc);
    SceneRecords r = s->rec;                                     // the records the new tree is built over (not owned)
    if (newVerts) r.verts = newVerts;
    const uint32_t n = s->tree.info.nLeaf, nNode = 2 * n - 1;
    {
        trq::PoolScratch mem(s->device, nullptr);
        RefBVH* leaves = nullptr;
        if ((rc = trq::reachable_leaves_on_device(s->tree.bvh, s->tree.ref, s->tree.info.nNode, n, r.verts, r.idx, mem, &leaves)) != TRQ_OK) return bail(rc);
        if (pool_malloc((void**)&t.bvh, (size_t)nNode * sizeof(RefBVH)) != cudaSuccess)
            return bail(trq::fail(TRQ_ERR_NOMEM, "trq_scene_rebuild: out of device memory"));
        if (n == 1) {                                            // the lone leaf is the root (BVH.hh:52-54), parent 0
            cudaError_t e = cudaMemcpyAsync(t.bvh, leaves, sizeof(RefBVH), cudaMemcpyDeviceToDevice, nullptr);
            if (e != cudaSuccess) return bail(trq::fail(TRQ_ERR_CUDA, "trq_scene_rebuild: %s", cudaGetErrorString(e)));
        } else {
            uint32_t depth = 0;
            rc = (flags & TRQ_BUILD_MORTON) ? trq::build_morton_on_device(leaves, n, t.bvh, s->device, &depth)
                                            : trq::build_on_device(leaves, n, t.bvh, s->device, &depth);
            if (rc == TRQ_ERR_DEPTH)
                return bail(trq::fail(TRQ_ERR_DEPTH, "trq_scene_rebuild: the new tree has interior depth %u, above the 32-bit trail's 31 "
                                                     "(Render.hh:140); the scene is unchanged", depth));
            if (rc != TRQ_OK) return bail(rc);
        }
    }
    if ((rc = plan_tree(t, nNode, r, s->device, "trq_scene_rebuild")) != TRQ_OK) return bail(rc);
    if ((rc = pack_tree(t, r, s->device)) != TRQ_OK) return bail(rc);

    // commit: the new tree (and vertices) in, the old ones out
    s->treeTraced.store(false);
    std::swap(s->tree, t);
    t.release();
    if (newVerts) { pool_free(s->rec.verts); s->rec.verts = newVerts; }
    if (!(s->userCfg && s->tree.cfg[s->defaultCfg].usable)) { s->defaultCfg = s->tree.autoCfg; s->userCfg = false; }
    return TRQ_OK;
}

int trq_scene_copy_bvh(const trq_scene* s, void* out, uint32_t flags) {
    if (!s || !out) return trq::fail(TRQ_ERR_INVALID, "trq_scene_copy_bvh: NULL argument");
    DeviceGuard guard(s->device);
    if (!guard.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", s->device);
    TRQ_CUDA(cudaMemcpy(out, s->tree.bvh, (size_t)s->tree.info.nNode * sizeof(RefBVH), (flags & TRQ_HOST_PTRS) ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice));
    return TRQ_OK;
}

int trq_scene_destroy(trq_scene* s) {
    if (!s) return TRQ_OK;
    DeviceGuard guard(s->device);
    free_scene(s);
    return TRQ_OK;
}

int trq_device_trim(int device) {
    cudaMemPool_t pool = trq::scratch_pool(device);
    if (!pool) return trq::fail(TRQ_ERR_CUDA, "trq_device_trim: no pool for device %d", device);
    DeviceGuard guard(device);
    TRQ_CUDA(cudaDeviceSynchronize());
    TRQ_CUDA(cudaMemPoolTrimTo(pool, 0));
    return TRQ_OK;
}

int trq_kernel_config_count(void) { return kNumCfgs; }

const char* trq_kernel_config_name(int cfg) { return (cfg >= 0 && cfg < kNumCfgs) ? kCfgs[cfg].name : nullptr; }

int trq_scene_set_kernel_config(trq_scene* s, int cfg, uint32_t* topNodesStaged) {
    if (!s) return trq::fail(TRQ_ERR_INVALID, "trq_scene_set_kernel_config: NULL scene");
    const bool user = cfg >= 0;
    if (cfg < 0) cfg = s->tree.autoCfg;
    if (cfg >= kNumCfgs) return trq::fail(TRQ_ERR_INVALID, "trq_scene_set_kernel_config: %d configurations", kNumCfgs);
    if (!s->tree.cfg[cfg].usable) return trq::fail(TRQ_ERR_INVALID, "trq_scene_set_kernel_config: configuration %s does not fit this scene (stack depth %u)", kCfgs[cfg].name, s->tree.stackDepth);
    s->defaultCfg = cfg;
    s->userCfg = user;
    if (topNodesStaged) *topNodesStaged = kCfgs[cfg].top ? s->tree.cfg[cfg].topCount : 0;
    return TRQ_OK;
}

int trq_scene_kernel_config(const trq_scene* s) { return s ? pick_cfg(s) : -1; }

int trq_scene_info(const trq_scene* s, trq_scene_info_t* info) {
    if (!s || !info) return trq::fail(TRQ_ERR_INVALID, "trq_scene_info: NULL argument");
    *info = s->tree.info;
    return TRQ_OK;
}

int trq_profile_enable(trq_scene* s, int on) {
    if (!s) return trq::fail(TRQ_ERR_INVALID, "trq_profile_enable: NULL scene");
    DeviceGuard guard(s->device);
    if (on && !s->evProf[0][0]) {
        for (int k = 0; k < kProfRing; ++k)
            for (int j = 0; j < 3; ++j) TRQ_CUDA(cudaEventCreate(&s->evProf[k][j]));
        TRQ_CUDA(cudaMalloc((void**)&s->d_profStamps, 2 * kProfRing * sizeof(unsigned long long)));
    }
    std::lock_guard<std::mutex> lock(s->profMutex);
    s->profile = on != 0;
    s->profHead = 0; s->profCount = 0;
    return TRQ_OK;
}

int trq_profile_read(trq_scene* s, uint32_t* nLaunches, float* traceMs, float* resolveMs) {
    if (!s || !nLaunches || !traceMs || !resolveMs) return trq::fail(TRQ_ERR_INVALID, "trq_profile_read: NULL argument");
    DeviceGuard guard(s->device);
    std::lock_guard<std::mutex> lock(s->profMutex);
    *nLaunches = 0; *traceMs = 0.0f; *resolveMs = 0.0f;
    // early launches: the time during which at least one of them ran (they overlap their predecessors by design)
    std::vector<std::pair<unsigned long long, unsigned long long>> spans;
    for (uint32_t k = 0; k < s->profCount; ++k) {
        if (!s->profByKernel[(s->profHead - 1 - k) % kProfRing]) continue;
        if (spans.empty()) {
            TRQ_CUDA(cudaDeviceSynchronize());
            std::vector<unsigned long long> h(2 * kProfRing);
            TRQ_CUDA(cudaMemcpy(h.data(), s->d_profStamps, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
            for (uint32_t j = 0; j < s->profCount; ++j) {
                const uint32_t slot = (s->profHead - 1 - j) % kProfRing;
                if (s->profByKernel[slot]) spans.emplace_back(h[2 * slot], h[2 * slot + 1]);
            }
            std::sort(spans.begin(), spans.end());
            unsigned long long covered = 0, reach = 0;
            for (const auto& sp : spans) {
                const unsigned long long from = sp.first > reach ? sp.first : reach;
                if (sp.second > from) covered += sp.second - from;
                if (sp.second > reach) reach = sp.second;
            }
            *traceMs += (float)(covered * 1e-6);
        }
        (*nLaunches)++;
    }
    for (uint32_t k = 0; k < s->profCount; ++k) {
        if (s->profByKernel[(s->profHead - 1 - k) % kProfRing]) continue;
        cudaEvent_t* ev = s->evProf[(s->profHead - 1 - k) % kProfRing];
        TRQ_CUDA(cudaEventSynchronize(ev[2]));
        float a = 0.0f, b = 0.0f;
        TRQ_CUDA(cudaEventElapsedTime(&a, ev[0], ev[1]));
        TRQ_CUDA(cudaEventElapsedTime(&b, ev[1], ev[2]));
        *traceMs += a; *resolveMs += b; (*nLaunches)++;
    }
    s->profHead = 0; s->profCount = 0;
    return TRQ_OK;
}

int trq_trace(trq_scene* s, const trq_ray* rays, uint64_t n, uint32_t flags, void* hits, void* stream) {
    if (!s) return trq::fail(TRQ_ERR_INVALID, "trq_trace: NULL scene");
    if (n == 0) return TRQ_OK;
    if (!rays || !hits) return trq::fail(TRQ_ERR_INVALID, "trq_trace: NULL rays/hits");
    if ((flags & TRQ_HIT16) && s->tree.maxPIndex >= (1u << 28))
        return trq::fail(TRQ_ERR_INVALID, "trq_trace: TRQ_HIT16 packs pIndex into 28 bits; this scene has pIndex up to %u", s->tree.maxPIndex);
    if (!(flags & TRQ_HOST_PTRS) && ((((uintptr_t)rays) & 31u) || (((uintptr_t)hits) & ((flags & TRQ_HIT16) ? 15u : 31u))))
        return trq::fail(TRQ_ERR_INVALID, "trq_trace: device rays / hits must be aligned to their record size (32 / 32 or 16 bytes: one access per record)");
    DeviceGuard guard(s->device);
    if (!guard.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", s->device);
    if (flags & TRQ_HOST_PTRS) return trace_host(s, rays, n, flags, hits);
    return launch_trace(s, rays, n, flags, hits, (cudaStream_t)stream);
}

int trq_host_sync(trq_scene* s) {
    if (!s) return trq::fail(TRQ_ERR_INVALID, "trq_host_sync: NULL scene");
    DeviceGuard guard(s->device);
    std::lock_guard<std::mutex> lock(s->stageMutex);
    return sync_staging(s);
}

int trq_expand_hits(trq_scene* s, const trq_ray* rays, const trq_hit* hits, uint64_t n, uint32_t flags,
                    trq_hit_record* records, void* stream) {
    if (!s) return trq::fail(TRQ_ERR_INVALID, "trq_expand_hits: NULL scene");
    if (n == 0) return TRQ_OK;
    if (!rays || !hits || !records) return trq::fail(TRQ_ERR_INVALID, "trq_expand_hits: NULL argument");
    DeviceGuard guard(s->device);
    if (!guard.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", s->device);
    const unsigned block = 256;
    const uint64_t grid = (n + block - 1) / block;
    if (flags & TRQ_HOST_PTRS) {
        trq_ray* dr = nullptr; trq_hit* dh = nullptr; trq_hit_record* dq = nullptr;
        TRQ_CUDA(cudaMalloc((void**)&dr, n * sizeof(trq_ray)));
        if (cudaMalloc((void**)&dh, n * sizeof(trq_hit)) != cudaSuccess) { cudaFree(dr); return trq::fail(TRQ_ERR_CUDA, "cudaMalloc failed"); }
        if (cudaMalloc((void**)&dq, n * sizeof(trq_hit_record)) != cudaSuccess) { cudaFree(dr); cudaFree(dh); return trq::fail(TRQ_ERR_CUDA, "cudaMalloc failed"); }
        cudaError_t e = cudaMemcpy(dr, rays, n * sizeof(trq_ray), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(dh, hits, n * sizeof(trq_hit), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) { expand_hits_kernel<<<(unsigned)grid, block>>>(scene_dev(s), dr, dh, dq, n); g_launches++; e = cudaGetLastError(); }
        if (e == cudaSuccess) e = cudaMemcpy(records, dq, n * sizeof(trq_hit_record), cudaMemcpyDeviceToHost);
        cudaFree(dr); cudaFree(dh); cudaFree(dq);
        if (e != cudaSuccess) return trq::fail(TRQ_ERR_CUDA, "trq_expand_hits: %s", cudaGetErrorString(e));
        return TRQ_OK;
    }
    expand_hits_kernel<<<(unsigned)grid, block, 0, (cudaStream_t)stream>>>(scene_dev(s), rays, hits, records, n);
    g_launches++;
    TRQ_CUDA(cudaGetLastError());
    return TRQ_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// Wavefront callers (SURVEY.md section 8, row f-3): device-side ray producers + a trace whose batch size lives
// on the device, so that cast -> trace -> spawn -> trace -> ... runs without a host round trip.
#include "../../include/tracer_rq_harness.h"
#include "kernels/producers.cuh"

extern "C" {

int trq_trace_indirect(trq_scene* s, const trq_ray* rays, const uint64_t* d_count, uint64_t capacity, uint32_t flags,
                       trq_hit* hits, void* stream) {
    if (!s) return trq::fail(TRQ_ERR_INVALID, "trq_trace_indirect: NULL scene");
    if (flags & TRQ_HOST_PTRS) return trq::fail(TRQ_ERR_INVALID, "trq_trace_indirect: device pointers only");
    if (capacity == 0) return TRQ_OK;
    if (!rays || !hits || !d_count) return trq::fail(TRQ_ERR_INVALID, "trq_trace_indirect: NULL argument");
    if ((((uintptr_t)rays) | ((uintptr_t)hits)) & 31u)
        return trq::fail(TRQ_ERR_INVALID, "trq_trace_indirect: rays/hits must be 32-byte aligned");
    DeviceGuard guard(s->device);
    if (!guard.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", s->device);
    return launch_trace(s, rays, capacity, flags, hits, (cudaStream_t)stream, (const unsigned long long*)d_count);
}

int trq_cast_rays(trq_scene* s, const trq_camera* cam, uint32_t W, uint32_t H, trq_ray* rays, void* stream) {
    if (!s || !cam || !rays) return trq::fail(TRQ_ERR_INVALID, "trq_cast_rays: NULL argument");
    if (cam->aperture != 0.0f) return trq::fail(TRQ_ERR_INVALID, "trq_cast_rays: only aperture 0 (the reference's setting, Tracer.mm:380) is supported");
    if ((uint64_t)W * H == 0) return TRQ_OK;
    DeviceGuard guard(s->device);
    if (!guard.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", s->device);
    float c[18];
    trqh_make_camera(cam->lookFrom, cam->lookAt, cam->viewUp, cam->vfov, cam->aspect, cam->focus_dist, c);   // MakeCamera, host
    CameraDev cd;
    for (int k = 0; k < 3; ++k) {
        cd.lookFrom[k] = c[k]; cd.u[k] = c[3 + k]; cd.v[k] = c[6 + k];
        cd.vertical[k] = c[9 + k]; cd.horizontal[k] = c[12 + k]; cd.corner[k] = c[15 + k];
    }
    cd.lenRadius = cam->aperture / 2;
    const uint64_t n = (uint64_t)W * H;
    cast_rays_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(cd, W, H, rays);
    g_launches++;
    TRQ_CUDA(cudaGetLastError());
    return TRQ_OK;
}

static int spawn_common(trq_scene* s, const trq_ray* rays, const trq_hit* hits, uint64_t n, const uint64_t* d_n,
                        uint64_t* d_count, const char* who) {
    if (!s) return trq::fail(TRQ_ERR_INVALID, "%s: NULL scene", who);
    if (!d_count) return trq::fail(TRQ_ERR_INVALID, "%s: NULL d_count", who);
    if (n && (!rays || !hits)) return trq::fail(TRQ_ERR_INVALID, "%s: NULL rays/hits", who);
    if (n > (1ull << 32)) return trq::fail(TRQ_ERR_INVALID, "%s: more than 2^32 rays in one call", who);

    return TRQ_OK;
}

int trq_spawn_bounce(trq_scene* s, const trq_ray* rays, const trq_hit* hits, uint64_t n, const uint64_t* d_n, uint64_t seedBase,
                     trq_ray* out, uint32_t* srcIndex, uint64_t* d_count, void* stream) {
    return trq_spawn_bounce_rng(s, rays, hits, n, d_n, seedBase, nullptr, nullptr, out, srcIndex, d_count, stream);
}

int trq_spawn_bounce_rng(trq_scene* s, const trq_ray* rays, const trq_hit* hits, uint64_t n, const uint64_t* d_n, uint64_t seedBase,
                         const uint32_t* pixelOf, uint32_t* rngState, trq_ray* out, uint32_t* srcIndex, uint64_t* d_count, void* stream) {
    int rc = spawn_common(s, rays, hits, n, d_n, d_count, "trq_spawn_bounce");
    if (rc == TRQ_OK && rngState && (((uintptr_t)rngState) & 15u)) rc = trq::fail(TRQ_ERR_INVALID, "trq_spawn_bounce_rng: rngState must be 16-byte aligned");
    if (rc != TRQ_OK) return rc;
    if (n && !out) return trq::fail(TRQ_ERR_INVALID, "trq_spawn_bounce: NULL out");
    DeviceGuard guard(s->device);
    if (!guard.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", s->device);
    cudaStream_t st = (cudaStream_t)stream;
    TRQ_CUDA(cudaMemsetAsync(d_count, 0, sizeof(uint64_t), st));
    if (n == 0) return TRQ_OK;
    spawn_bounce_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(scene_dev(s), rays, hits, n, (const unsigned long long*)d_n, seedBase, pixelOf, rngState, out, srcIndex,
                                                                      (unsigned long long*)d_count);

    g_launches++;
    TRQ_CUDA(cudaGetLastError());
    return TRQ_OK;
}

int trq_rng_frame_begin(trq_scene* s, uint32_t* rngState, uint64_t nPixels, void* stream) {
    if (!s) return trq::fail(TRQ_ERR_INVALID, "trq_rng_frame_begin: NULL scene");
    if (nPixels == 0) return TRQ_OK;
    if (!rngState || (((uintptr_t)rngState) & 15u)) return trq::fail(TRQ_ERR_INVALID, "trq_rng_frame_begin: rngState must be a 16-byte aligned device pointer");
    DeviceGuard guard(s->device);
    if (!guard.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", s->device);
    rng_frame_begin_kernel<<<(unsigned)((nPixels + 255) / 256), 256, 0, (cudaStream_t)stream>>>((uint4*)rngState, nPixels);
    g_launches++;
    TRQ_CUDA(cudaGetLastError());
    return TRQ_OK;
}

int trq_spawn_shadow(trq_scene* s, const trq_ray* rays, const trq_hit* hits, uint64_t n, const uint64_t* d_n, uint64_t seedBase,
                     uint32_t lightA, uint32_t lightB, trq_ray* out, uint32_t* srcIndex, uint64_t* d_count, void* stream) {
    return trq_spawn_shadow_rng(s, rays, hits, n, d_n, seedBase, nullptr, nullptr, lightA, lightB, out, srcIndex, d_count, stream);
}

int trq_spawn_shadow_rng(trq_scene* s, const trq_ray* rays, const trq_hit* hits, uint64_t n, const uint64_t* d_n, uint64_t seedBase,
                         const uint32_t* pixelOf, uint32_t* rngState, uint32_t lightA, uint32_t lightB, trq_ray* out, uint32_t* srcIndex,
                         uint64_t* d_count, void* stream) {
    int rc = spawn_common(s, rays, hits, n, d_n, d_count, "trq_spawn_shadow");
    if (rc == TRQ_OK && rngState && (((uintptr_t)rngState) & 15u)) rc = trq::fail(TRQ_ERR_INVALID, "trq_spawn_shadow_rng: rngState must be 16-byte aligned");
    if (rc != TRQ_OK) return rc;
    if (n && !out) return trq::fail(TRQ_ERR_INVALID, "trq_spawn_shadow: NULL out");
    if (lightA >= s->tree.info.nSquare || lightB >= s->tree.info.nSquare)
        return trq::fail(TRQ_ERR_INVALID, "trq_spawn_shadow: light index out of range (nSquare %u)", s->tree.info.nSquare);
    DeviceGuard guard(s->device);
    if (!guard.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", s->device);
    cudaStream_t st = (cudaStream_t)stream;
    TRQ_CUDA(cudaMemsetAsync(d_count, 0, sizeof(uint64_t), st));
    if (n == 0) return TRQ_OK;
    spawn_shadow_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(scene_dev(s), rays, hits, n, (const unsigned long long*)d_n, seedBase, pixelOf, rngState, lightA, lightB, out, srcIndex,
                                                                      (unsigned long long*)d_count);
    g_launches++;
    TRQ_CUDA(cudaGetLastError());
    return TRQ_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// Peer-memory hit gather (SURVEY.md section 8e: a consumer that wants every rank's hits whole). One process per GPU;
// every rank owns a buffer [phase][rank][capacity] of trq_hit plus a small header (flags, counts), exported through
// CUDA IPC. trq_trace_gather traces this rank's rays into slot [rank] of its own buffer and, BESIDE the trace kernel,
// runs a sender kernel on a second stream: the trace counts finished records per tile of 2^TRQ_GATHER_TILE_SHIFT
// records (default 2^11 = 2048), the sender ships each complete tile into slot [rank] of EVERY other rank's buffer over
// NVLink (gather_send_tma_kernel with TMA bulk copies; gather_send_kernel with coalesced 16-byte stores when
// TRQ_GATHER_TMA=0 or when the TMA sender's staging does not fit beside the trace CTAs). The
// all-gather runs under the traversal, tile by tile, with no NCCL call; the sender's last CTA publishes (count, step)
// with system-scope release stores. trq_gather_wait enqueues a small kernel that acquires all ranks' step numbers.
// Three phases (step mod 3): a peer can start writing phase p again at step k + 3 only after it has seen this rank's
// flag for step k + 2, so the result of step k stays valid until this rank's trq_trace_gather for step k + 2 executes.
namespace {
constexpr size_t kGatherHeader = 4096;                 // flags[16] u64 @0, counts[3][16] u64 @128
constexpr size_t kGatherCountsAt = 128;
constexpr unsigned kGatherPhases = 3;
}

struct trq_gather {
    trq_scene* scene = nullptr;
    uint32_t rank = 0, world = 1;
    uint64_t capacity = 0;
    uint8_t* base = nullptr;
    uint8_t* peerBase[TRQ_GATHER_MAX_RANKS] = {};
    unsigned int* h_status = nullptr;                  // pinned + mapped: raised by gather_wait_kernel on timeout
    unsigned int* d_status = nullptr;
    unsigned long long step = 0;
    uint32_t lastFlags = 0;
    bool connected = false;
    cudaStream_t sendStream = nullptr;                 // gather_send_kernel runs here, beside the trace on the caller's stream
    cudaEvent_t evStart = nullptr, evSent = nullptr;
    uint32_t* d_tileDone = nullptr;                    // finished records per tile of the step being traced
    unsigned int* d_blocksDone = nullptr;
    int numSMs = 0;
    size_t slot_offset(unsigned phase, uint32_t r) const {
        return kGatherHeader + ((size_t)phase * world + r) * capacity * sizeof(trq_hit);
    }
};

extern "C" {

int trq_gather_create(trq_scene* s, uint32_t rank, uint32_t world, uint64_t capacity, trq_gather** out, void* handle) {
    if (!s || !out || !handle) return trq::fail(TRQ_ERR_INVALID, "trq_gather_create: NULL argument");
    *out = nullptr;
    if (world == 0 || world > TRQ_GATHER_MAX_RANKS || rank >= world)
        return trq::fail(TRQ_ERR_INVALID, "trq_gather_create: rank %u / world %u (at most %d ranks)", rank, world, TRQ_GATHER_MAX_RANKS);
    if (capacity == 0 || capacity > (1ull << 31)) return trq::fail(TRQ_ERR_INVALID, "trq_gather_create: capacity out of range");
    static_assert(sizeof(cudaIpcMemHandle_t) == TRQ_GATHER_HANDLE_BYTES, "IPC handle size");
    DeviceGuard guard(s->device);
    if (!guard.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", s->device);
    trq_gather* g = new (std::nothrow) trq_gather();
    if (!g) return trq::fail(TRQ_ERR_NOMEM, "trq_gather_create: out of host memory");
    g->scene = s; g->rank = rank; g->world = world; g->capacity = capacity;
    const size_t total = kGatherHeader + (size_t)kGatherPhases * world * capacity * sizeof(trq_hit);
    cudaError_t e = cudaMalloc((void**)&g->base, total);
    if (e == cudaSuccess) e = cudaMemset(g->base, 0, kGatherHeader);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaHostAlloc((void**)&g->h_status, sizeof(unsigned int), cudaHostAllocMapped);
    if (e == cudaSuccess) { *g->h_status = 0; e = cudaHostGetDevicePointer((void**)&g->d_status, g->h_status, 0); }
    const size_t nTiles = (size_t)((capacity + (1ull << TRQ_GATHER_TILE_SHIFT_MIN) - 1) >> TRQ_GATHER_TILE_SHIFT_MIN);
    if (e == cudaSuccess) e = cudaMalloc((void**)&g->d_tileDone, (nTiles + 1) * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemset(g->d_tileDone, 0, (nTiles + 1) * sizeof(uint32_t));   // last word: blocksDone
    if (e == cudaSuccess) { g->d_blocksDone = g->d_tileDone + nTiles; e = cudaStreamCreateWithFlags(&g->sendStream, cudaStreamNonBlocking); }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g->evStart, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g->evSent, cudaEventDisableTiming);
    g->numSMs = s->numSMs;
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, g->base);
    if (e != cudaSuccess) {
        cudaFree(g->base); cudaFree(g->d_tileDone); if (g->h_status) cudaFreeHost(g->h_status);
        if (g->sendStream) cudaStreamDestroy(g->sendStream);
        if (g->evStart) cudaEventDestroy(g->evStart);
        if (g->evSent) cudaEventDestroy(g->evSent);
        delete g;
        return trq::fail(TRQ_ERR_CUDA, "trq_gather_create (%zu bytes): %s", total, cudaGetErrorString(e));
    }
    memcpy(handle, &h, sizeof h);
    *out = g;
    return TRQ_OK;
}

int trq_gather_connect(trq_gather* g, const void* handles) {
    if (!g || (!handles && g->world > 1)) return trq::fail(TRQ_ERR_INVALID, "trq_gather_connect: NULL argument");
    if (g->connected) return trq::fail(TRQ_ERR_INVALID, "trq_gather_connect: already connected");
    DeviceGuard guard(g->scene->device);
    for (uint32_t r = 0; r < g->world; ++r) {
        if (r == g->rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const uint8_t*)handles + (size_t)r * sizeof h, sizeof h);
        cudaError_t e = cudaIpcOpenMemHandle((void**)&g->peerBase[r], h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess)
            return trq::fail(TRQ_ERR_CUDA, "trq_gather_connect: cudaIpcOpenMemHandle(rank %u) failed: %s (one process per GPU, same node)",
                             r, cudaGetErrorString(e));
    }
    g->connected = true;
    return TRQ_OK;
}

int trq_trace_gather(trq_scene* s, trq_gather* g, const trq_ray* rays, uint64_t n, uint32_t flags, void* stream) {
    if (!s || !g || g->scene != s) return trq::fail(TRQ_ERR_INVALID, "trq_trace_gather: NULL or foreign scene / gather");
    if (!g->connected) return trq::fail(TRQ_ERR_INVALID, "trq_trace_gather: call trq_gather_connect first");
    if (flags & (TRQ_HOST_PTRS | TRQ_HOST_ASYNC | TRQ_KERNEL_REFLAYOUT)) return trq::fail(TRQ_ERR_INVALID, "trq_trace_gather: device pointers and the packed kernel only");
    if (n > g->capacity) return trq::fail(TRQ_ERR_INVALID, "trq_trace_gather: %llu rays exceed the capacity %llu", (unsigned long long)n, (unsigned long long)g->capacity);
    if (n && !rays) return trq::fail(TRQ_ERR_INVALID, "trq_trace_gather: NULL rays");
    if (((uintptr_t)rays) & 31u) return trq::fail(TRQ_ERR_INVALID, "trq_trace_gather: rays must be 32-byte aligned");
    if ((flags & TRQ_HIT16) && s->tree.maxPIndex >= (1u << 28)) return trq::fail(TRQ_ERR_INVALID, "trq_trace_gather: TRQ_HIT16 packs pIndex into 28 bits");
    DeviceGuard guard(s->device);
    if (!guard.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", s->device);
    const unsigned long long step = ++g->step;
    const unsigned phase = (unsigned)(step % kGatherPhases);
    g->lastFlags = flags;
    static const unsigned long long timeoutNs = [] {
        const char* e = getenv("TRQ_GATHER_TIMEOUT_MS");
        return (unsigned long long)(e ? atoll(e) : 10000) * 1000000ull;
    }();
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* own = g->base + g->slot_offset(phase, g->rank);
    SendParams G{};
    G.src = (const uint4*)own;
    G.n = n; G.step = step; G.timeoutNs = timeoutNs;
    G.unitsPerRecord = (flags & TRQ_HIT16) ? 1u : 2u;
    G.tileDone = g->d_tileDone; G.blocksDone = g->d_blocksDone; G.status = g->d_status;
    G.ownFlag = (unsigned long long*)g->base + g->rank;
    G.ownCount = (unsigned long long*)(g->base + kGatherCountsAt) + phase * TRQ_GATHER_MAX_RANKS + g->rank;
    for (uint32_t r = 0; r < g->world; ++r) {
        if (r == g->rank) continue;
        const uint32_t k = G.nPeer++;
        G.peer[k] = (uint4*)(g->peerBase[r] + g->slot_offset(phase, g->rank));
        G.peerFlag[k] = (unsigned long long*)g->peerBase[r] + g->rank;
        G.peerCount[k] = (unsigned long long*)(g->peerBase[r] + kGatherCountsAt) + phase * TRQ_GATHER_MAX_RANKS + g->rank;
    }
    // records per tile: small tiles follow the trace closely (short tail after its last ray), large ones cost fewer polls
    static const uint32_t tileShift = [] {
        const char* e = getenv("TRQ_GATHER_TILE_SHIFT");
        int v = e ? atoi(e) : 11;
        return (uint32_t)(v < (int)TRQ_GATHER_TILE_SHIFT_MIN ? (int)TRQ_GATHER_TILE_SHIFT_MIN : (v > 16 ? 16 : v));
    }();
    G.tileShift = tileShift;
    const uint64_t nTiles = (n + (1ull << tileShift) - 1) >> tileShift;
    // the sender starts when the caller's stream reaches this point (its counters zeroed), runs beside the trace, and the
    // caller's stream continues after both
    if (nTiles) TRQ_CUDA(cudaMemsetAsync(g->d_tileDone, 0, nTiles * sizeof(uint32_t), st));
    TRQ_CUDA(cudaEventRecord(g->evStart, st));
    TRQ_CUDA(cudaStreamWaitEvent(g->sendStream, g->evStart, 0));
    unsigned sendGrid = (unsigned)g->numSMs;
    if (nTiles < sendGrid) sendGrid = nTiles ? (unsigned)nTiles : 1u;
    // The sender CTA (no shared memory of its own, 1 KB of per-CTA reserve) must fit beside the resident trace CTAs. The
    // driver sizes the SM's shared-memory carve-out to what the trace needs, rounded up to a supported size; when that leaves
    // less than the reserve (C3's depth: 5 x 39 KB = 195 of 196 KB), ask for the next size for this launch.
    const bool any = (flags & TRQ_TRACE_ANY) != 0, hit16 = (flags & TRQ_HIT16) != 0;
    const void* fn = kCfgs[0].fn[s->tree.leaves][any ? 1 : 0][hit16 ? 1 : 0];
    bool bumped = false, useTma = false;
    size_t chosen = 228 * 1024;
    if (n) {
        static const size_t kCarveKB[] = {0, 8, 16, 32, 64, 100, 132, 164, 196, 228};
        const size_t need = (size_t)s->tree.cfg[0].blocksPerSM[any ? 1 : 0][hit16 ? 1 : 0] * (s->tree.cfg[0].smem + kSmemBlockReserve);
        for (size_t kb : kCarveKB) if (kb * 1024 >= need) { chosen = kb * 1024; break; }
        static const int tmaEnv = [] { const char* e = getenv("TRQ_GATHER_TMA"); return e ? atoi(e) : 1; }();
        // the TMA sender stages through 24 KB of shared memory; beside a trace that leaves less than that even at the largest
        // carve-out (very deep trees) the LSU sender, which needs none, is the one that can run concurrently
        useTma = tmaEnv != 0 && 228 * 1024 >= need + kSmemBlockReserve + 512 + (size_t)TRQ_SEND_TMA_STAGES * TRQ_SEND_TMA_CHUNK + 256;
        const size_t senderSmem = useTma ? (size_t)TRQ_SEND_TMA_STAGES * TRQ_SEND_TMA_CHUNK + 256 : 0;
        const bool bump = chosen - need < kSmemBlockReserve + 512 + senderSmem && chosen < 228 * 1024;
        if (bump)
            for (size_t kb : kCarveKB) if (kb * 1024 > chosen) { chosen = kb * 1024; break; }
        const int carveout = (int)((chosen * 100 + kSmemPerSM - 1) / kSmemPerSM);
        // The sender may reach an SM before the trace does: it starts with the caller's stream at evStart, and with
        // TRQ_SORT_RAYS the ordering kernels still run ahead of the trace. An SM takes its carve-out from the first CTA it
        // gets, and the sender's own need (24 KB, or none) leaves no room for a trace CTA. With a sender CTA on every SM
        // (nTiles >= numSMs) the trace then has nowhere to run and every sender waits for the timeout. The sender asks for
        // the trace's carve-out, so a trace CTA fits beside it whichever kernel arrives first.
        TRQ_CUDA(cudaFuncSetAttribute(useTma ? (const void*)gather_send_tma_kernel : (const void*)gather_send_kernel,
                                      cudaFuncAttributePreferredSharedMemoryCarveout, carveout));
        if (bump) bumped = cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, carveout) == cudaSuccess;
    }
    const int rc = launch_trace(s, rays, n, flags, own, st, nullptr, g->d_tileDone, tileShift);     // first: its CTAs take their places
    if (bumped) cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutDefault);
    if (rc != TRQ_OK) return rc;
    if (useTma) gather_send_tma_kernel<<<sendGrid, 32, TRQ_SEND_TMA_STAGES * TRQ_SEND_TMA_CHUNK, g->sendStream>>>(G);
    else        gather_send_kernel<<<sendGrid, 128, 0, g->sendStream>>>(G);
    g_launches++;
    TRQ_CUDA(cudaGetLastError());
    TRQ_CUDA(cudaEventRecord(g->evSent, g->sendStream));
    TRQ_CUDA(cudaStreamWaitEvent(st, g->evSent, 0));
    return TRQ_OK;
}

int trq_gather_wait(trq_gather* g, void* stream, const void** hitsAll, const uint64_t** counts) {
    if (!g) return trq::fail(TRQ_ERR_INVALID, "trq_gather_wait: NULL gather");
    if (g->step == 0) return trq::fail(TRQ_ERR_INVALID, "trq_gather_wait: nothing traced yet");
    DeviceGuard guard(g->scene->device);
    static const unsigned long long timeoutNs = [] {
        const char* e = getenv("TRQ_GATHER_TIMEOUT_MS");
        return (unsigned long long)(e ? atoll(e) : 10000) * 1000000ull;
    }();
    gather_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((const unsigned long long*)g->base, g->world, g->step, timeoutNs, g->d_status);
    g_launches++;
    TRQ_CUDA(cudaGetLastError());
    const unsigned phase = (unsigned)(g->step % kGatherPhases);
    if (hitsAll) *hitsAll = g->base + g->slot_offset(phase, 0);
    if (counts) *counts = (const uint64_t*)(g->base + kGatherCountsAt) + phase * TRQ_GATHER_MAX_RANKS;
    return TRQ_OK;
}

int trq_gather_status(trq_gather* g) {
    if (!g) return trq::fail(TRQ_ERR_INVALID, "trq_gather_status: NULL gather");
    const unsigned int v = *(volatile unsigned int*)g->h_status;
    if (v & 0x80000000u) return trq::fail(TRQ_ERR_CUDA, "trq_trace_gather: the trace did not finish a tile before the timeout");
    if (v) return trq::fail(TRQ_ERR_CUDA, "trq_gather_wait: rank %u did not publish its hits before the timeout", v - 1);
    return TRQ_OK;
}

int trq_gather_destroy(trq_gather* g) {
    if (!g) return TRQ_OK;
    DeviceGuard guard(g->scene->device);
    cudaDeviceSynchronize();
    for (uint32_t r = 0; r < g->world; ++r) if (g->peerBase[r]) cudaIpcCloseMemHandle(g->peerBase[r]);
    if (g->sendStream) cudaStreamDestroy(g->sendStream);
    if (g->evStart) cudaEventDestroy(g->evStart);
    if (g->evSent) cudaEventDestroy(g->evSent);
    cudaFree(g->d_tileDone);
    cudaFree(g->base);
    if (g->h_status) cudaFreeHost(g->h_status);
    delete g;
    return TRQ_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// Single-process multi-GPU helper (SURVEY.md section 8b "multi-GPU helper trq_mgpu_* owns one scene per rank", 8e): the
// reference's host is ONE process, so this is the form of ray sharding it can adopt without a launcher: one scene per
// device, host rays cut into contiguous ranges [k*n/R, (k+1)*n/R), every device's range staged and traced through its
// own copy engines and streams at once (TRQ_HOST_ASYNC on every scene, then one wait per scene). No collective anywhere:
// the scene is replicated by uploading it R times, the hits land in the caller's host array.
struct trq_mgpu {
    std::vector<trq_scene*> scenes;
};

extern "C" {

int trq_mgpu_create(const trq_scene_desc* desc, const int* devices, int nDevices, trq_mgpu** out) {
    if (!desc || !out) return trq::fail(TRQ_ERR_INVALID, "trq_mgpu_create: NULL argument");
    *out = nullptr;
    const int have = trq_device_count();
    if (have <= 0) return trq::fail(TRQ_ERR_NO_DEVICE, "trq_mgpu_create: no CUDA device (there is no CPU fallback)");
    if (nDevices <= 0) nDevices = have;                        // all visible devices
    if (nDevices > have && !devices) return trq::fail(TRQ_ERR_INVALID, "trq_mgpu_create: %d devices requested, %d visible", nDevices, have);
    trq_mgpu* m = new (std::nothrow) trq_mgpu();
    if (!m) return trq::fail(TRQ_ERR_NOMEM, "trq_mgpu_create: out of host memory");
    for (int k = 0; k < nDevices; ++k) {
        trq_scene* s = nullptr;
        const int rc = trq_scene_create(desc, devices ? devices[k] : k, &s);
        if (rc != TRQ_OK) {
            for (trq_scene* t : m->scenes) trq_scene_destroy(t);
            delete m;
            return rc;
        }
        m->scenes.push_back(s);
    }
    *out = m;
    return TRQ_OK;
}

int trq_mgpu_device_count(const trq_mgpu* m) { return m ? (int)m->scenes.size() : 0; }

trq_scene* trq_mgpu_scene(trq_mgpu* m, int k) {
    if (!m || k < 0 || k >= (int)m->scenes.size()) { trq::fail(TRQ_ERR_INVALID, "trq_mgpu_scene: index out of range"); return nullptr; }
    return m->scenes[k];
}

int trq_mgpu_shard(const trq_mgpu* m, uint64_t n, int k, uint64_t* lo, uint64_t* hi) {
    if (!m || !lo || !hi || k < 0 || k >= (int)m->scenes.size()) return trq::fail(TRQ_ERR_INVALID, "trq_mgpu_shard: bad argument");
    const unsigned __int128 R = m->scenes.size();
    *lo = (uint64_t)((unsigned __int128)n * (unsigned)k / R);
    *hi = (uint64_t)((unsigned __int128)n * (unsigned)(k + 1) / R);
    return TRQ_OK;
}

int trq_mgpu_trace(trq_mgpu* m, const trq_ray* rays, uint64_t n, uint32_t flags, void* hits) {
    if (!m) return trq::fail(TRQ_ERR_INVALID, "trq_mgpu_trace: NULL handle");
    if (n == 0) return TRQ_OK;
    if (!rays || !hits) return trq::fail(TRQ_ERR_INVALID, "trq_mgpu_trace: NULL rays/hits");
    const size_t recBytes = (flags & TRQ_HIT16) ? sizeof(trq_hit16) : sizeof(trq_hit);
    int first = TRQ_OK;
    for (int k = 0; k < (int)m->scenes.size(); ++k) {           // queue every device's range ...
        uint64_t lo, hi;
        trq_mgpu_shard(m, n, k, &lo, &hi);
        if (hi == lo) continue;
        const int rc = trq_trace(m->scenes[k], rays + lo, hi - lo, flags | TRQ_HOST_PTRS | TRQ_HOST_ASYNC, (uint8_t*)hits + lo * recBytes, nullptr);
        if (rc != TRQ_OK && first == TRQ_OK) first = rc;
    }
    for (trq_scene* s : m->scenes) {                            // ... then wait for all of them
        const int rc = trq_host_sync(s);
        if (rc != TRQ_OK && first == TRQ_OK) first = rc;
    }
    return first;
}

int trq_mgpu_destroy(trq_mgpu* m) {
    if (!m) return TRQ_OK;
    for (trq_scene* s : m->scenes) trq_scene_destroy(s);
    delete m;
    return TRQ_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// Memory-system probes for the roofline report (SURVEY.md section 8d: "no L2 figure is in MEASURED_PEAKS.json, so the
// harness must measure it"): read-only 16-byte loads that bypass L1 (ld.global.cg) over a working set that fits in L2
// (32 MB) or does not (2 GB), all SMs, best of five.
namespace {
__global__ void __launch_bounds__(256)
probe_read_kernel(const uint4* __restrict__ buf, uint64_t n16, int iters, uint32_t* sink) {
    uint32_t acc = 0;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (int it = 0; it < iters; ++it)
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride) {
            const uint4 v = __ldcg(buf + i);
            acc += v.x ^ v.y ^ v.z ^ v.w;
        }
    if (acc == 0x12345678u) *sink = acc;          // keeps the loads alive
}
}  // namespace

extern "C" int trq_probe_bandwidth(int device, int which, double* gbs) {
    if (!gbs) return trq::fail(TRQ_ERR_INVALID, "trq_probe_bandwidth: NULL argument");
    int ndev = trq_device_count();
    if (ndev <= 0) return trq::fail(TRQ_ERR_NO_DEVICE, "trq_probe_bandwidth: no CUDA device");
    if (device < 0 || device >= ndev) return trq::fail(TRQ_ERR_INVALID, "trq_probe_bandwidth: device out of range");
    DeviceGuard guard(device);
    cudaDeviceProp prop;
    TRQ_CUDA(cudaGetDeviceProperties(&prop, device));
    const uint64_t bytes = which == 0 ? (32ull << 20) : (2ull << 30);
    const int iters = which == 0 ? 64 : 2;
    uint4* buf = nullptr; uint32_t* sink = nullptr;
    TRQ_CUDA(cudaMalloc((void**)&buf, bytes));
    if (cudaMalloc((void**)&sink, 4) != cudaSuccess) { cudaFree(buf); return trq::fail(TRQ_ERR_CUDA, "cudaMalloc failed"); }
    cudaMemset(buf, 1, bytes);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    const unsigned grid = (unsigned)prop.multiProcessorCount * 8u;
    float best = 1e30f;
    for (int rep = 0; rep < 6; ++rep) {
        cudaEventRecord(e0);
        probe_read_kernel<<<grid, 256>>>(buf, bytes / 16, iters, sink);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms = 0.0f; cudaEventElapsedTime(&ms, e0, e1);
        if (rep > 0 && ms < best) best = ms;
        g_launches++;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaError_t e = cudaGetLastError();
    cudaFree(buf); cudaFree(sink);
    if (e != cudaSuccess) return trq::fail(TRQ_ERR_CUDA, "trq_probe_bandwidth: %s", cudaGetErrorString(e));
    *gbs = (double)bytes * iters / (best * 1e-3) / 1e9;
    return TRQ_OK;
}
