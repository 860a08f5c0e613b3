// tracer_b200/csrc/bvh_build_gpu.cu -- BVH::buildTree (BVH.hh:246-269) on the GPU.
//   trq_bvh_build_tree_device   leaves and result in DEVICE memory (feeds trq_scene_create_device without a host round trip)
//   trq_bvh_build_tree_gpu      the same build for a HOST array (copy in, build, copy out)
//   trq_bvh_build_tree_morton_device   the Morton-order builder (kernels/morton_build.cuh), DEVICE memory
//   trq_bvh_build_nodes_triangles_device / trq_bvh_build_nodes_device   BVH::buildNode per primitive (kernels/leaves.cuh)
// Orchestrates the level-synchronous kernels of kernels/bvh_build.cuh; same node array as trq_bvh_build_tree.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <vector>

#include "../../include/tracer_rq.h"
#include "host/error.h"
#include "host/gpu_build.h"
#include "host/layout.h"
#include "host/scratch.h"
#include "kernels/bvh_build.cuh"
#include "kernels/leaves.cuh"
#include "kernels/morton_build.cuh"

#include <cub/device/device_radix_sort.cuh>

using namespace trq;
using namespace trq::gpubuild;

namespace trq {
void note_launches(uint64_t n);

// One stream-ordered pool per device that keeps its memory between calls: scratch for the builder and for scene
// creation comes back without a cudaMalloc after the first use.
cudaMemPool_t scratch_pool(int device) {
    static std::mutex m;
    static std::map<int, cudaMemPool_t> pools;
    std::lock_guard<std::mutex> lock(m);
    auto it = pools.find(device);
    if (it != pools.end()) return it->second;
    cudaMemPoolProps pp = {};
    pp.allocType = cudaMemAllocationTypePinned;
    pp.handleTypes = cudaMemHandleTypeNone;
    pp.location.type = cudaMemLocationTypeDevice;
    pp.location.id = device;
    cudaMemPool_t pool = nullptr;
    if (cudaMemPoolCreate(&pool, &pp) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    unsigned long long keep = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    pools[device] = pool;
    return pool;
}

}  // namespace trq

namespace {

#define BCK(call)                                                                                   \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        if (e_ != cudaSuccess)                                                                      \
            return trq::fail(TRQ_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

inline unsigned blocks(uint64_t n, unsigned b) { return (unsigned)((n + b - 1) / b); }

struct DeviceScope {
    int prev = -1;
    bool ok = false;
    explicit DeviceScope(int dev) { cudaGetDevice(&prev); ok = cudaSetDevice(dev) == cudaSuccess; }
    ~DeviceScope() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace

// Interior depth above 31 still builds, refits and reports the whole tree, then returns TRQ_ERR_DEPTH as the host
// builder does. *maxDepthOut is written only when the tree is complete; the callers set it to 0 first.
int trq::build_on_device(const RefBVH* dLeaves, uint32_t n, RefBVH* dOut, int device, uint32_t* maxDepthOut) {
    const uint32_t nNode = 2 * n - 1;
    cudaStream_t st = nullptr;                          // legacy default stream: ordered with the caller's cudaMemcpy / kernels
    PoolScratch mem(device, st);
    uint32_t *idx, *seg, *flag, *scanT, *tileSums, *fallbackList, *arrivals, *counters;
    unsigned long long* sortKeys;                       // the fallback's sort keys; outside it, the two swap lists
    float4* cen;
    BNode *tabA, *tabB;
    const uint32_t cap = n / 2 + 1;
    const uint32_t nTiles = blocks((uint64_t)n + 1, kScanTile);
    bool ok = mem.alloc(&idx, n) && mem.alloc(&seg, n) &&
              mem.alloc(&flag, (size_t)n + 1) && mem.alloc(&scanT, (size_t)n + 1) && mem.alloc(&tileSums, nTiles) &&
              mem.alloc(&sortKeys, n) && mem.alloc(&fallbackList, cap) && mem.alloc(&arrivals, nNode) &&
              mem.alloc(&counters, 4) && mem.alloc(&cen, n) && mem.alloc(&tabA, cap) && mem.alloc(&tabB, cap);
    if (!ok) return trq::fail(TRQ_ERR_NOMEM, "BVH build on the GPU: out of device memory");
    uint32_t* leftFalse = reinterpret_cast<uint32_t*>(sortKeys);
    uint32_t* rightTrue = leftFalse + n;

    BCK(cudaMemsetAsync(dOut, 0, (size_t)nNode * sizeof(RefBVH), st));
    BCK(cudaMemcpyAsync(dOut + 1, dLeaves, (size_t)n * sizeof(RefBVH), cudaMemcpyDeviceToDevice, st));     // leaves at 1..N (BVH.hh:265)
    BCK(cudaMemsetAsync(arrivals, 0, (size_t)nNode * sizeof(uint32_t), st));
    BCK(cudaMemsetAsync(counters, 0, 4 * sizeof(uint32_t), st));
    uint64_t launches = 0;
    init_elements_kernel<<<blocks(n, 256), 256, 0, st>>>(dLeaves, n, idx, seg, cen); ++launches;
    BNode root; std::memset(&root, 0, sizeof root);
    root.start = 0; root.end = n; root.base = 0;
    BCK(cudaMemcpyAsync(tabA, &root, sizeof root, cudaMemcpyHostToDevice, st));
    BCK(cudaStreamSynchronize(st));                     // `root` lives on this stack frame

    BNode *cur = tabA, *nxt = tabB;
    uint32_t nActive = 1, depth = 0;
    uint32_t* nNext = counters;          // [0] next-level count, [1] max depth, [2] level-table overflow, [3] fallback nodes
    uint32_t* dMaxDepth = counters + 1;
    uint32_t* dOverflow = counters + 2;
    uint32_t* nFallback = counters + 3;
    while (nActive > 0) {
        // every split leaves both children strictly smaller than their parent, so level n - 2 is the deepest possible
        if (depth > n - 2) return trq::fail(TRQ_ERR_LAYOUT, "BVH build on the GPU: internal: level %u of %u leaves", depth, n);
        reset_nodes_kernel<<<blocks(nActive, 256), 256, 0, st>>>(cur, nActive, nFallback);
        centroid_bounds_kernel<<<blocks(n, 256), 256, 0, st>>>(idx, seg, cen, n, cur);
        choose_axis_kernel<<<blocks(nActive, 256), 256, 0, st>>>(cur, nActive);
        bucket_kernel<<<blocks(n, 256), 256, 0, st>>>(dLeaves, idx, seg, cen, n, cur);
        choose_split_kernel<<<blocks(nActive, 128), 128, 0, st>>>(cur, nActive);
        predicate_kernel<<<blocks((uint64_t)n + 1, 256), 256, 0, st>>>(idx, seg, cen, n, cur, flag);
        scan_tiles_kernel<<<nTiles, 1024, 0, st>>>(flag, scanT, n + 1, tileSums);
        scan_sums_kernel<<<1, 1024, 0, st>>>(tileSums, nTiles);
        scan_add_kernel<<<nTiles, 1024, 0, st>>>(scanT, n + 1, tileSums);
        midpoint_kernel<<<blocks(nActive, 256), 256, 0, st>>>(cur, nActive, scanT, fallbackList, nFallback);
        mispl_kernel<<<blocks(n, 256), 256, 0, st>>>(seg, n, cur, flag, scanT, leftFalse, rightTrue);
        swap_kernel<<<blocks(n, 256), 256, 0, st>>>(seg, n, cur, leftFalse, rightTrue, idx);
        fallback_sort_kernel<<<kSortBlocks, kSortThreads, 0, st>>>(cur, fallbackList, nFallback, cen, idx, sortKeys);   // exits at once without fallback nodes
        BCK(cudaMemsetAsync(nNext, 0, sizeof(uint32_t), st));
        emit_kernel<<<blocks(nActive, 128), 128, 0, st>>>(cur, nActive, idx, cen, dOut, n, nxt, cap, nNext, dOverflow, dMaxDepth, depth);
        reseg_kernel<<<blocks(n, 256), 256, 0, st>>>(seg, n, cur);
        launches += 15;
        uint32_t lvl[3] = {0, 0, 0};
        BCK(cudaMemcpyAsync(lvl, counters, sizeof lvl, cudaMemcpyDeviceToHost, st));
        BCK(cudaStreamSynchronize(st));
        nActive = lvl[0];
        if (lvl[2] || nActive > cap) return trq::fail(TRQ_ERR_LAYOUT, "BVH build on the GPU: internal: level table overflow");
        BNode* t = cur; cur = nxt; nxt = t;
        ++depth;
    }
    refit_kernel<<<blocks(n, 256), 256, 0, st>>>(dOut, n, arrivals); ++launches;
    uint32_t maxDepth = 0;
    BCK(cudaMemcpyAsync(&maxDepth, dMaxDepth, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    BCK(cudaStreamSynchronize(st));
    BCK(cudaGetLastError());
    trq::note_launches(launches);
    if (maxDepthOut) *maxDepthOut = maxDepth;
    if (maxDepth > 31)
        return trq::fail(TRQ_ERR_DEPTH, "BVH build on the GPU: interior depth %u exceeds the 32-bit trail (Render.hh:140)", maxDepth);
    return TRQ_OK;
}

// The Morton builder (kernels/morton_build.cuh): bounds, codes, CUB's radix sort of (code, position) -- stable, and the
// positions enter in order, so ties stay in list order -- 32 split launches whose counts stay on the device, the shared
// refit, and one read of the depth at the end. Never TRQ_ERR_DEPTH: the depth clamp bounds every tree at 31.
int trq::build_morton_on_device(const RefBVH* dLeaves, uint32_t n, RefBVH* dOut, int device, uint32_t* maxDepthOut) {
    using namespace trq::morton;
    const uint32_t nNode = 2 * n - 1;
    cudaStream_t st = nullptr;
    PoolScratch mem(device, st);
    uint64_t *codeA, *codeB;
    uint32_t *posA, *posB, *counters, *arrivals;
    Open *tabA, *tabB;
    Bounds* bounds;
    const uint32_t cap = n / 2 + 1;
    size_t sortBytes = 0;
    cub::DoubleBuffer<uint64_t> keys(nullptr, nullptr);
    cub::DoubleBuffer<uint32_t> vals(nullptr, nullptr);
    BCK(cub::DeviceRadixSort::SortPairs(nullptr, sortBytes, keys, vals, (int)n, 0, 63, st));
    uint8_t* sortTemp;
    bool ok = mem.alloc(&codeA, n) && mem.alloc(&codeB, n) && mem.alloc(&posA, n) && mem.alloc(&posB, n) &&
              mem.alloc(&counters, (size_t)kCounters + nNode) && mem.alloc(&tabA, cap) && mem.alloc(&tabB, cap) &&
              mem.alloc(&bounds, 1) && mem.alloc(&sortTemp, sortBytes);
    if (!ok) return trq::fail(TRQ_ERR_NOMEM, "Morton BVH build on the GPU: out of device memory");
    arrivals = counters + kCounters;

    int sms = 0;
    BCK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    const unsigned grid = std::min(blocks(cap, 256), (unsigned)sms * 4u);
    BCK(cudaMemcpyAsync(dOut + 1, dLeaves, (size_t)n * sizeof(RefBVH), cudaMemcpyDeviceToDevice, st));     // leaves at 1..n
    BCK(cudaMemsetAsync(counters, 0, ((size_t)kCounters + nNode) * sizeof(uint32_t), st));
    morton_init_kernel<<<1, 32, 0, st>>>(bounds, tabA, n, counters);
    morton_bounds_kernel<<<std::min(blocks(n, 256), (unsigned)sms * 8u), 256, 0, st>>>(dLeaves, n, bounds);
    morton_code_kernel<<<blocks(n, 256), 256, 0, st>>>(dLeaves, n, bounds, codeA, posA);
    keys = cub::DoubleBuffer<uint64_t>(codeA, codeB);
    vals = cub::DoubleBuffer<uint32_t>(posA, posB);
    BCK(cub::DeviceRadixSort::SortPairs(sortTemp, sortBytes, keys, vals, (int)n, 0, 63, st));
    Open *cur = tabA, *nxt = tabB;
    for (uint32_t depth = 0; depth < kMaxLevels; ++depth) {
        morton_level_kernel<<<grid, 256, 0, st>>>(keys.Current(), vals.Current(), n, cur, nxt, cap, counters, depth, dOut);
        std::swap(cur, nxt);
    }
    gpubuild::refit_kernel<<<blocks(n, 256), 256, 0, st>>>(dOut, n, arrivals);
    // 3 + 32 + 1 launches of ours; CUB's onesweep sort: a histogram, a scan and one launch per 8-bit digit
    trq::note_launches(36 + 2 + 8);
    uint32_t tail[2] = {0, 0};                          // deepest level, overflow flag
    BCK(cudaMemcpyAsync(tail, counters + kMaxDepth, sizeof tail, cudaMemcpyDeviceToHost, st));
    BCK(cudaStreamSynchronize(st));
    BCK(cudaGetLastError());
    if (tail[1]) return trq::fail(TRQ_ERR_LAYOUT, "Morton BVH build on the GPU: internal: level table overflow");
    if (maxDepthOut) *maxDepthOut = tail[0];
    return TRQ_OK;
}

// flag -> exclusive scan (the builder's scan kernels) -> scatter
int trq::reachable_leaves_on_device(const RefBVH* bvh, const uint32_t* ref, uint32_t nNode, uint32_t nLeaf, const RefVertex* verts,
                                    const uint32_t* idx, PoolScratch& mem, RefBVH** leavesOut) {
    cudaStream_t st = nullptr;
    const uint32_t nTiles = blocks((uint64_t)nNode + 1, kScanTile);
    uint32_t *flag, *pos, *tileSums;
    if (!(mem.alloc(&flag, (size_t)nNode + 1) && mem.alloc(&pos, (size_t)nNode + 1) && mem.alloc(&tileSums, nTiles) && mem.alloc(leavesOut, nLeaf)))
        return trq::fail(TRQ_ERR_NOMEM, "trq_scene_rebuild: out of device memory");
    leaves::reachable_leaf_flag_kernel<<<blocks((uint64_t)nNode + 1, 256), 256, 0, st>>>(bvh, ref, nNode, flag);
    scan_tiles_kernel<<<nTiles, 1024, 0, st>>>(flag, pos, nNode + 1, tileSums);
    scan_sums_kernel<<<1, 1024, 0, st>>>(tileSums, nTiles);
    scan_add_kernel<<<nTiles, 1024, 0, st>>>(pos, nNode + 1, tileSums);
    leaves::reachable_leaf_scatter_kernel<<<blocks(nNode, 256), 256, 0, st>>>(bvh, flag, pos, nNode, verts, idx, *leavesOut);
    trq::note_launches(5);
    BCK(cudaGetLastError());
    return TRQ_OK;
}

int trq::refit_primitive_leaves_on_device(RefBVH* bvh, const uint32_t* ref, uint32_t nNode, const RefSphere* spheres, const RefSquare* squares,
                                          const RefCube* cubes) {
    leaves::RecordLists lists = {};
    const void* list[3] = {spheres, squares, cubes};
    for (int32_t t = TRQ_SPHERE; t <= TRQ_CUBE; ++t) {
        leaves::RecordList& r = lists.kind[t];
        r.list = (const uint8_t*)list[t];
        leaves::record_layout(t, &r.stride, &r.modelAt, &r.boxAt);
    }
    leaves::refit_primitive_leaves_kernel<<<blocks(nNode, 256), 256>>>(bvh, ref, nNode, lists);
    trq::note_launches(1);
    BCK(cudaGetLastError());
    return TRQ_OK;
}

namespace {

int check_device(int device, const char* who) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); return trq::fail(TRQ_ERR_NO_DEVICE, "%s: no CUDA device (use trq_bvh_build_tree on the host)", who); }
    if (device < 0 || device >= ndev) return trq::fail(TRQ_ERR_INVALID, "%s: device %d out of range", who, device);
    return TRQ_OK;
}

}  // namespace

extern "C" int trq_bvh_build_tree_device(void* d_bvhList, uint32_t nLeaves, int device, uint32_t* nNodeOut, uint32_t* maxDepthOut) {
    if (maxDepthOut) *maxDepthOut = 0;
    if (!d_bvhList || nLeaves == 0) return trq::fail(TRQ_ERR_INVALID, "trq_bvh_build_tree_device: empty leaf list");
    if (nLeaves > 0x3fffffffu) return trq::fail(TRQ_ERR_INVALID, "trq_bvh_build_tree_device: too many leaves");
    int rc = check_device(device, "trq_bvh_build_tree_device");
    if (rc != TRQ_OK) return rc;
    DeviceScope scope(device);
    if (!scope.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    RefBVH* d = (RefBVH*)d_bvhList;
    const uint32_t n = nLeaves;
    if (nNodeOut) *nNodeOut = 2 * n - 1;
    if (n == 1) {                                   // BVH.hh:52-54 + :263-268: the lone leaf becomes node 0
        BCK(cudaMemset(&d[0].parent, 0, sizeof(uint32_t)));
        if (maxDepthOut) *maxDepthOut = 0;
        return TRQ_OK;
    }
    // the result overwrites the leaves' slots (they move to 1..n), so the build reads a copy of them
    PoolScratch mem(device, nullptr);
    RefBVH* dLeaves = nullptr;
    if (!mem.alloc(&dLeaves, n)) return trq::fail(TRQ_ERR_NOMEM, "trq_bvh_build_tree_device: out of device memory");
    BCK(cudaMemcpyAsync(dLeaves, d, (size_t)n * sizeof(RefBVH), cudaMemcpyDeviceToDevice, nullptr));
    return build_on_device(dLeaves, n, d, device, maxDepthOut);
}

extern "C" int trq_bvh_build_tree_morton_device(void* d_bvhList, uint32_t nLeaves, int device, uint32_t* nNodeOut, uint32_t* maxDepthOut) {
    if (maxDepthOut) *maxDepthOut = 0;
    if (!d_bvhList || nLeaves == 0) return trq::fail(TRQ_ERR_INVALID, "trq_bvh_build_tree_morton_device: empty leaf list");
    if (nLeaves > 0x3fffffffu) return trq::fail(TRQ_ERR_INVALID, "trq_bvh_build_tree_morton_device: too many leaves");
    int rc = check_device(device, "trq_bvh_build_tree_morton_device");
    if (rc != TRQ_OK) return rc;
    DeviceScope scope(device);
    if (!scope.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    RefBVH* d = (RefBVH*)d_bvhList;
    const uint32_t n = nLeaves;
    if (nNodeOut) *nNodeOut = 2 * n - 1;
    if (n == 1) {                                   // the lone leaf becomes node 0, as trq_bvh_build_tree_device does
        BCK(cudaMemset(&d[0].parent, 0, sizeof(uint32_t)));
        return TRQ_OK;
    }
    PoolScratch mem(device, nullptr);               // the result overwrites the leaves' slots: build from a copy
    RefBVH* dLeaves = nullptr;
    if (!mem.alloc(&dLeaves, n)) return trq::fail(TRQ_ERR_NOMEM, "trq_bvh_build_tree_morton_device: out of device memory");
    BCK(cudaMemcpyAsync(dLeaves, d, (size_t)n * sizeof(RefBVH), cudaMemcpyDeviceToDevice, nullptr));
    return build_morton_on_device(dLeaves, n, d, device, maxDepthOut);
}

extern "C" int trq_bvh_build_tree_gpu(void* bvhList, uint32_t nLeaves, int device, uint32_t* nNodeOut, uint32_t* maxDepthOut) {
    if (maxDepthOut) *maxDepthOut = 0;
    if (!bvhList || nLeaves == 0) return trq::fail(TRQ_ERR_INVALID, "trq_bvh_build_tree_gpu: empty leaf list");
    if (nLeaves > 0x3fffffffu) return trq::fail(TRQ_ERR_INVALID, "trq_bvh_build_tree_gpu: too many leaves");
    const uint32_t n = nLeaves, nNode = 2 * n - 1;
    RefBVH* host = (RefBVH*)bvhList;
    if (n == 1) {                                   // BVH.hh:52-54 + :263-268: the lone leaf becomes node 0
        host[0].parent = 0;
        if (nNodeOut) *nNodeOut = 1;
        if (maxDepthOut) *maxDepthOut = 0;
        return TRQ_OK;
    }
    int rc = check_device(device, "trq_bvh_build_tree_gpu");
    if (rc != TRQ_OK) return rc;
    DeviceScope scope(device);
    if (!scope.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    PoolScratch mem(device, nullptr);
    RefBVH *dLeaves = nullptr, *dOut = nullptr;
    if (!mem.alloc(&dLeaves, n) || !mem.alloc(&dOut, nNode)) return trq::fail(TRQ_ERR_NOMEM, "trq_bvh_build_tree_gpu: out of device memory");
    BCK(cudaMemcpyAsync(dLeaves, host, (size_t)n * sizeof(RefBVH), cudaMemcpyHostToDevice, nullptr));
    uint32_t maxDepth = 0;
    rc = build_on_device(dLeaves, n, dOut, device, &maxDepth);
    if (nNodeOut) *nNodeOut = nNode;
    if (maxDepthOut) *maxDepthOut = maxDepth;
    if (rc != TRQ_OK && rc != TRQ_ERR_DEPTH) return rc;
    BCK(cudaMemcpy(host, dOut, (size_t)nNode * sizeof(RefBVH), cudaMemcpyDeviceToHost));
    return rc;
}

extern "C" int trq_bvh_build_nodes_triangles_device(const void* d_triList, const uint32_t* d_idxList, uint32_t nTri, uint32_t pIndexBase,
                                                    void* d_nodes_out, int device, void* stream) {
    if (nTri == 0) return TRQ_OK;
    if (!d_triList || !d_idxList || !d_nodes_out) return trq::fail(TRQ_ERR_INVALID, "trq_bvh_build_nodes_triangles_device: NULL argument");
    int rc = check_device(device, "trq_bvh_build_nodes_triangles_device");
    if (rc != TRQ_OK) return rc;
    DeviceScope scope(device);
    if (!scope.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    leaves::triangle_leaves_kernel<<<blocks(nTri, 256), 256, 0, (cudaStream_t)stream>>>((const RefVertex*)d_triList, d_idxList, nTri,
                                                                                     pIndexBase, (RefBVH*)d_nodes_out);
    trq::note_launches(1);
    BCK(cudaGetLastError());
    return TRQ_OK;
}

extern "C" int trq_bvh_build_nodes_device(int32_t pType, const void* d_list, uint32_t n, uint32_t pIndexBase, void* d_nodes_out,
                                          int device, void* stream) {
    uint32_t stride, modelAt, boxAt;
    if (!leaves::record_layout(pType, &stride, &modelAt, &boxAt))
        return trq::fail(TRQ_ERR_INVALID, "trq_bvh_build_nodes_device: pType %d is not TRQ_SPHERE, TRQ_SQUARE or TRQ_CUBE", pType);
    if (n == 0) return TRQ_OK;
    if (!d_list || !d_nodes_out) return trq::fail(TRQ_ERR_INVALID, "trq_bvh_build_nodes_device: NULL argument");
    int rc = check_device(device, "trq_bvh_build_nodes_device");
    if (rc != TRQ_OK) return rc;
    DeviceScope scope(device);
    if (!scope.ok) return trq::fail(TRQ_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    leaves::primitive_leaves_kernel<<<blocks(n, 256), 256, 0, (cudaStream_t)stream>>>((const uint8_t*)d_list, n, stride, modelAt, boxAt, pType,
                                                                                   pIndexBase, (RefBVH*)d_nodes_out);
    trq::note_launches(1);
    BCK(cudaGetLastError());
    return TRQ_OK;
}
