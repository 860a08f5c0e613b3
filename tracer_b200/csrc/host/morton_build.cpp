// tracer_b200/csrc/host/morton_build.cpp
//
// The Morton-order builder restated on the host: sequential, strict fp32 (-ffp-contract=off), the rules of
// kernels/morton_build.cuh step by step. It is the pin the device builder (trq_bvh_build_tree_morton_device) is tested
// against byte for byte, and hosts without a GPU can build with it.

#include "../../../include/tracer_rq.h"
#include "error.h"
#include "layout.h"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstring>
#include <exception>
#include <vector>

namespace {

using trq::RefBVH;

constexpr uint32_t kQuantMax = (1u << 21) - 1;

// AABB::centroid  AABB.hh:22-25 :  mini + (maxi - mini) / 2
inline void centroid_of(const RefBVH& n, float c[3]) {
    for (int k = 0; k < 3; ++k) c[k] = n.bBOX.mini[k] + (n.bBOX.maxi[k] - n.bBOX.mini[k]) / 2;
}

// morton::quantise, operation for operation
inline uint32_t quantise(float c, float lo, float hi) {
    if (std::isnan(c) || c == INFINITY) return kQuantMax;
    if (c == -INFINITY) return 0u;
    const float ext = hi - lo;
    if (!(lo <= hi) || !(std::isfinite(ext) && ext > 0.0f)) return 0u;
    const float q = std::floor(((c - lo) / ext) * 2097152.0f);
    return q >= (float)kQuantMax ? kQuantMax : (uint32_t)q;
}

// CUDA's fminf / fmaxf, which gpubuild::refit_kernel uses: a NaN operand is ignored, and -0.0 orders below +0.0 whichever
// operand it is (the host's fminf returns its second operand when the two compare equal)
inline float min_box(float a, float b) { return (a == 0.0f && b == 0.0f) ? (std::signbit(a) ? a : b) : fminf(a, b); }
inline float max_box(float a, float b) { return (a == 0.0f && b == 0.0f) ? (std::signbit(a) ? b : a) : fmaxf(a, b); }

inline uint64_t spread3(uint32_t v) {                       // bit i -> bit 3i
    uint64_t x = 0;
    for (int i = 0; i < 21; ++i) x |= (uint64_t)((v >> i) & 1u) << (3 * i);
    return x;
}

struct Morton {
    RefBVH* nodes;                  // final layout
    const uint64_t* code;           // by sorted position
    const uint32_t* order;          // list position of each sorted position
    uint32_t n, gRoot;

    // left size and axis of the node over sorted [a, b] at depth d
    void split(uint32_t a, uint32_t b, uint32_t d, uint32_t* s, uint32_t* axis) const {
        const uint32_t m = b - a + 1;
        const uint64_t ca = code[a], cb = code[b];
        if (ca == cb) {
            *s = m / 2;
            *axis = 0;
        } else {
            int h = 63;
            while (!(((ca ^ cb) >> h) & 1u)) --h;
            *axis = 2u - (uint32_t)h % 3u;
            // positions with bit h clear come first (sorted, common prefix above h); code[a] has it clear, code[b] set
            const uint64_t* p = std::partition_point(code + a + 1, code + b, [h](uint64_t c) { return !((c >> h) & 1u); });
            *s = (uint32_t)(p - (code + a));
        }
        const uint64_t lim = 1ull << (31 - d);              // depth clamp
        uint64_t lo = m > lim ? m - lim : 0, hi = lim;
        lo = std::max<uint64_t>(lo, 1);
        hi = std::min<uint64_t>(hi, m - 1);
        *s = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(*s, lo), hi);
    }

    uint32_t index_of(uint32_t g) const { return g < gRoot ? n + 1 + g : n + g; }

    // emits the subtree over sorted [a, b] as node `self` (its gap already chosen), returns the deepest interior level
    uint32_t emit(uint32_t a, uint32_t b, uint32_t d, uint32_t self, uint32_t parent, uint32_t s, uint32_t axis) {
        RefBVH nb;
        std::memset(&nb, 0, sizeof nb);
        nb.parent = parent;
        nb.axis = axis;
        nb.pType = TRQ_BVH;
        uint32_t deepest = d;
        const uint32_t span[2][2] = {{a, a + s - 1}, {a + s, b}};
        uint32_t child[2];
        for (int c = 0; c < 2; ++c) {
            const uint32_t ca = span[c][0], cb = span[c][1];
            if (ca == cb) {
                child[c] = 1 + order[ca];
                nodes[child[c]].parent = self;
            } else {
                uint32_t cs, caxis;
                split(ca, cb, d + 1, &cs, &caxis);
                child[c] = index_of(ca + cs - 1);
                deepest = std::max(deepest, emit(ca, cb, d + 1, child[c], self, cs, caxis));
            }
        }
        nb.left = child[0];
        nb.right = child[1];
        for (int k = 0; k < 3; ++k) {                       // AABB::make(box, box), as gpubuild::refit_kernel
            nb.bBOX.mini[k] = min_box(nodes[child[0]].bBOX.mini[k], nodes[child[1]].bBOX.mini[k]);
            nb.bBOX.maxi[k] = max_box(nodes[child[0]].bBOX.maxi[k], nodes[child[1]].bBOX.maxi[k]);
        }
        nodes[self] = nb;
        return deepest;
    }
};

}  // namespace

extern "C" int trq_bvh_build_tree_morton(void* bvhList, uint32_t nLeaves, uint32_t* nNodeOut, uint32_t* maxDepthOut) {
    if (maxDepthOut) *maxDepthOut = 0;
    if (!bvhList || nLeaves == 0) return trq::fail(TRQ_ERR_INVALID, "trq_bvh_build_tree_morton: empty leaf list");
    if (nLeaves > 0x3fffffffu) return trq::fail(TRQ_ERR_INVALID, "trq_bvh_build_tree_morton: too many leaves");
    RefBVH* nodes = (RefBVH*)bvhList;
    const uint32_t n = nLeaves, nNode = 2 * n - 1;
    if (nNodeOut) *nNodeOut = nNode;
    if (n == 1) {                                           // the lone leaf is node 0
        nodes[0].parent = 0;
        return TRQ_OK;
    }
    uint32_t maxDepth = 0;
    try {                                                   // no C++ exception may cross the C ABI
        std::vector<float> cen(3 * (size_t)n);
        float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
        for (uint32_t i = 0; i < n; ++i) {
            centroid_of(nodes[i], &cen[3 * (size_t)i]);
            for (int k = 0; k < 3; ++k) {
                const float v = cen[3 * (size_t)i + k];
                if (std::isfinite(v)) { lo[k] = std::min(lo[k], v); hi[k] = std::max(hi[k], v); }
            }
        }
        std::vector<uint64_t> key(n);
        std::vector<uint32_t> order(n);
        for (uint32_t i = 0; i < n; ++i) {
            const float* c = &cen[3 * (size_t)i];
            key[i] = spread3(quantise(c[0], lo[0], hi[0])) << 2 | spread3(quantise(c[1], lo[1], hi[1])) << 1 |
                     spread3(quantise(c[2], lo[2], hi[2]));
            order[i] = i;
        }
        std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return key[a] < key[b]; });
        std::vector<uint64_t> code(n);
        for (uint32_t p = 0; p < n; ++p) code[p] = key[order[p]];

        std::memmove(nodes + 1, nodes, sizeof(RefBVH) * (size_t)n);        // leaves at 1..n in list order (BVH.hh:265)
        Morton mb{nodes, code.data(), order.data(), n, 0};
        uint32_t s, axis;
        mb.split(0, n - 1, 0, &s, &axis);
        mb.gRoot = s - 1;
        maxDepth = mb.emit(0, n - 1, 0, 0, 0, s, axis);                    // recursion depth <= 32 (the depth clamp)
    } catch (const std::exception& e) {
        return trq::fail(TRQ_ERR_NOMEM, "trq_bvh_build_tree_morton: %s", e.what());
    }
    if (maxDepthOut) *maxDepthOut = maxDepth;
    return TRQ_OK;
}
