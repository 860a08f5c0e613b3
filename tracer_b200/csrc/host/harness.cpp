// tracer_b200/csrc/host/harness.cpp -- workload generators (see include/tracer_rq_harness.h).
//
// Host restatements of the reference's ray PRODUCERS, strict IEEE fp32 in the order the
// reference writes them (compile with -ffp-contract=off). File:line cites are to
// /root/reference/RT_Metal.

#include "../../../include/tracer_rq_harness.h"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstring>
#include <thread>
#include <vector>

#include "layout.h"

namespace {

constexpr float kPi = 3.14159265358979323846264338327950288f;   // M_PI_F

struct V3 { float x, y, z; };
inline V3 operator+(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
inline V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline V3 operator*(V3 a, float s) { return {a.x * s, a.y * s, a.z * s}; }
inline V3 operator*(float s, V3 a) { return {s * a.x, s * a.y, s * a.z}; }
inline V3 operator/(V3 a, float s) { return {a.x / s, a.y / s, a.z / s}; }
inline float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline V3 cross(V3 a, V3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
inline float length(V3 a) { return sqrtf(dot(a, a)); }
inline V3 normalize(V3 a) { return a / length(a); }
inline float get(V3 a, unsigned i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }
inline void set(V3& a, unsigned i, float v) { if (i == 0) a.x = v; else if (i == 1) a.y = v; else a.z = v; }

// Random.metal:3-25 (= pcg_basic.c:44-67)
struct Pcg32 {
    uint64_t state, inc;
    Pcg32(uint64_t initstate, uint64_t initseq) {
        state = 0u;
        inc = (initseq << 1u) | 1u;
        next();
        state += initstate;
        next();
    }
    uint32_t next() {
        uint64_t old = state;
        state = old * 6364136223846793005ULL + inc;
        uint32_t xorshifted = (uint32_t)(((old >> 18u) ^ old) >> 27u);
        uint32_t rot = (uint32_t)(old >> 59u);
        return (xorshifted >> rot) | (xorshifted << ((-rot) & 31));
    }
    float randomF() { return ldexpf((float)next(), -32); }            // Random.metal:21-26
    // the per-pixel state texture of the reference (RGBA32Uint) in exRNG's layout: r = state >> 32, g = state,
    // b = inc >> 32, a = inc, on load and store (toRNG's entry swap is trqh_rng_frame_begin, once per frame)
    struct Raw {};
    Pcg32(Raw, const uint32_t t[4]) {
        state = ((uint64_t)t[0] << 32) | t[1];
        inc = ((uint64_t)t[2] << 32) | t[3];
    }
    void store(uint32_t t[4]) const {                                 // exRNG  Render.hh:109-120
        t[0] = (uint32_t)(state >> 32); t[1] = (uint32_t)state; t[2] = (uint32_t)(inc >> 32); t[3] = (uint32_t)inc;
    }
};

// RNG of record i: the pixel's stored stream when a state texture is given, else PCG32(seedBase + i, 1).
struct RngSlot {
    Pcg32 rng;
    uint32_t* slot;
    uint32_t pixel;
    RngSlot(uint64_t seedBase, uint64_t i, const uint32_t* pixelOf, uint32_t* rngState)
        : rng(seedBase + i, 1), slot(nullptr), pixel(pixelOf ? pixelOf[i] : (uint32_t)i) {
        if (rngState) { slot = rngState + 4 * (size_t)pixel; rng = Pcg32(Pcg32::Raw{}, slot); }
    }
    ~RngSlot() { if (slot) rng.store(slot); }
};

// (int32_t)v as x86 computes it (cvttss2si), spelled out because the cast is undefined for NaN and out-of-range values:
// truncation toward zero, INT32_MIN for NaN and for values outside [-2^31, 2^31). The device uses the same rule.
inline int32_t x86_f2i(float v) { return (v != v || v >= 0x1p31f || v < -0x1p31f) ? INT32_MIN : (int32_t)v; }

// Math.hh:57-74; the negation and the add into the float's bits wrap modulo 2^32
inline V3 offset_ray(V3 p, V3 n) {
    const float origin = 1.0f / 32.0f, float_scale = 1.0f / 65536.0f, int_scale = 256.0f;
    float pin[3] = {p.x, p.y, p.z}, nin[3] = {n.x, n.y, n.z}, out[3];
    for (int k = 0; k < 3; ++k) {
        uint32_t of_i = (uint32_t)x86_f2i(int_scale * nin[k]);
        uint32_t pi; std::memcpy(&pi, &pin[k], 4);
        pi += (pin[k] < 0) ? 0u - of_i : of_i;
        float p_i; std::memcpy(&p_i, &pi, 4);
        out[k] = fabsf(pin[k]) < origin ? pin[k] + float_scale * nin[k] : p_i;
    }
    return {out[0], out[1], out[2]};
}

// Sampling.hh:18-34
inline void coordinate_system(V3 a, V3& b, V3& c) {
    if (fabsf(a.x) > fabsf(a.y)) b = {-a.z, 0.0f, a.x};
    else                         b = {0.0f, a.z, -a.y};
    b = normalize(b);
    c = cross(a, b);
}

// Sampling.hh:79-99
inline void concentric_sample_disk(float u0, float u1, float& dx, float& dy) {
    float ox = 2.f * u0 - 1.0f, oy = 2.f * u1 - 1.0f;
    if (ox == 0 && oy == 0) { dx = 0; dy = 0; return; }
    const float PiOver2 = kPi / 2.0f, PiOver4 = kPi / 4.0f;
    float theta, r;
    if (fabsf(ox) > fabsf(oy)) { r = ox; theta = PiOver4 * (oy / ox); }
    else                       { r = oy; theta = PiOver2 - PiOver4 * (ox / oy); }
    dx = r * cosf(theta); dy = r * sinf(theta);
}

// Sampling.hh:125-129
inline V3 cosine_sample_hemisphere(float u0, float u1) {
    float dx, dy;
    concentric_sample_disk(u0, u1, dx, dy);
    float z = sqrtf(fmaxf(0.0f, 1.0f - dx * dx - dy * dy));
    return {dx, dy, z};
}

template <typename F>
void parallel_for(uint64_t n, F f) {
    unsigned nt = std::max(1u, std::thread::hardware_concurrency());
    if (n < 65536) nt = 1;
    if (nt == 1) { f(0, n); return; }
    std::vector<std::thread> pool;
    for (unsigned k = 0; k < nt; ++k) pool.emplace_back(f, n * k / nt, n * (k + 1) / nt);
    for (auto& t : pool) t.join();
}

inline void store_ray(trq_ray& r, V3 o, V3 d, float tmax) {
    r.ox = o.x; r.oy = o.y; r.oz = o.z; r.tmax = tmax;
    r.dx = d.x; r.dy = d.y; r.dz = d.z; r.flags = 0;
}

}  // namespace

extern "C" {

void trqh_pcg32_fill_f32(uint64_t seed, uint64_t seq, uint64_t n, float* out) {
    Pcg32 rng(seed, seq);
    for (uint64_t i = 0; i < n; ++i) out[i] = rng.randomF();
}

void trqh_pcg32_fill_u32(uint64_t seed, uint64_t seq, uint64_t n, uint32_t* out) {
    Pcg32 rng(seed, seq);
    for (uint64_t i = 0; i < n; ++i) out[i] = rng.next();
}

void trqh_normalize_rays(trq_ray* rays, uint64_t n) {
    parallel_for(n, [&](uint64_t lo, uint64_t hi) {
        for (uint64_t i = lo; i < hi; ++i) {
            V3 d = normalize(V3{rays[i].dx, rays[i].dy, rays[i].dz});               // Ray.hh:21-23
            rays[i].dx = d.x; rays[i].dy = d.y; rays[i].dz = d.z;
        }
    });
}

void trqh_offset_ray(const float p[3], const float n[3], float out[3]) {
    V3 r = offset_ray(V3{p[0], p[1], p[2]}, V3{n[0], n[1], n[2]});
    out[0] = r.x; out[1] = r.y; out[2] = r.z;
}

void trqh_make_soup(uint32_t nTri, uint64_t seed, float extent, void* triList, uint32_t* idxList) {
    trq::RefVertex* tv = (trq::RefVertex*)triList;
    parallel_for(nTri, [&](uint64_t lo, uint64_t hi) {
        for (uint64_t i = lo; i < hi; ++i) {
            Pcg32 rng(seed, i);
            V3 c{rng.randomF(), rng.randomF(), rng.randomF()};
            V3 p[3];
            for (int k = 0; k < 3; ++k) {
                V3 xi{rng.randomF(), rng.randomF(), rng.randomF()};
                p[k] = {c.x + extent * (xi.x - 0.5f), c.y + extent * (xi.y - 0.5f), c.z + extent * (xi.z - 0.5f)};
            }
            V3 n = cross(p[1] - p[0], p[2] - p[0]);
            float len = length(n);
            n = len > 0 ? n / len : V3{0, 0, 1};
            for (int k = 0; k < 3; ++k) {
                trq::RefVertex& v = tv[3 * i + k];
                v.v[0] = p[k].x; v.v[1] = p[k].y; v.v[2] = p[k].z;
                v.n[0] = n.x; v.n[1] = n.y; v.n[2] = n.z;
                v.uv[0] = (k == 1) ? 1.0f : 0.0f; v.uv[1] = (k == 2) ? 1.0f : 0.0f;
                idxList[3 * i + k] = (uint32_t)(3 * i + k);
            }
        }
    });
}

void trqh_gen_random_rays(uint64_t first, uint64_t n, uint64_t seed, const float lo[3], const float hi[3],
                          float tmax, trq_ray* rays) {
    parallel_for(n, [&](uint64_t a, uint64_t b) {
        for (uint64_t i = a; i < b; ++i) {
            Pcg32 rng(seed, first + i);
            V3 o;
            o.x = lo[0] + (hi[0] - lo[0]) * rng.randomF();
            o.y = lo[1] + (hi[1] - lo[1]) * rng.randomF();
            o.z = lo[2] + (hi[2] - lo[2]) * rng.randomF();
            float z = 2.0f * rng.randomF() - 1.0f;
            float phi = 2.0f * kPi * rng.randomF();
            float r = sqrtf(fmaxf(0.0f, 1.0f - z * z));
            V3 d = normalize(V3{r * cosf(phi), r * sinf(phi), z});
            // keep every component away from exact zero (1/0 = inf slabs are legal but NaN-prone, SURVEY section 7)
            if (d.x == 0.0f) d.x = FLT_MIN;
            if (d.y == 0.0f) d.y = FLT_MIN;
            if (d.z == 0.0f) d.z = FLT_MIN;
            store_ray(rays[i], o, d, tmax);
        }
    });
}

void trqh_make_camera(const float lookFrom_[3], const float lookAt_[3], const float viewUp_[3],
                      float vfov, float aspect, float focus_dist, float out[18]) {
    // MakeCamera  Tracer.mm:87-125 (vfov in radians, passed straight through)
    V3 lookFrom{lookFrom_[0], lookFrom_[1], lookFrom_[2]}, lookAt{lookAt_[0], lookAt_[1], lookAt_[2]};
    V3 viewUp{viewUp_[0], viewUp_[1], viewUp_[2]};
    float theta = vfov;
    float halfHeight = tanf(theta / 2);
    float halfWidth = aspect * halfHeight;
    V3 w = normalize(lookFrom - lookAt);
    V3 u = normalize(cross(viewUp, w));
    V3 v = cross(w, u);
    V3 vertical = (2 * halfHeight * focus_dist) * v;
    V3 horizontal = (2 * halfWidth * focus_dist) * u;
    V3 corner = lookFrom - vertical / 2 - horizontal / 2 - focus_dist * w;
    const V3 all[6] = {lookFrom, u, v, vertical, horizontal, corner};
    for (int k = 0; k < 6; ++k) { out[3 * k] = all[k].x; out[3 * k + 1] = all[k].y; out[3 * k + 2] = all[k].z; }
}

void trqh_gen_camera_rays(const float lookFrom_[3], const float lookAt_[3], const float viewUp_[3],
                          float vfov, float aspect, float focus_dist, uint32_t W, uint32_t H, trq_ray* rays) {
    float cam[18];
    trqh_make_camera(lookFrom_, lookAt_, viewUp_, vfov, aspect, focus_dist, cam);
    const V3 lookFrom{cam[0], cam[1], cam[2]}, vertical{cam[9], cam[10], cam[11]}, horizontal{cam[12], cam[13], cam[14]},
             corner{cam[15], cam[16], cam[17]};
    parallel_for((uint64_t)W * H, [&](uint64_t a, uint64_t b) {
        for (uint64_t i = a; i < b; ++i) {
            uint32_t x = (uint32_t)(i % W), y = (uint32_t)(i / W);
            float s = float(x) / W, t = float(y) / H;                                // Render.metal:523-524
            V3 origin = lookFrom;                                                     // lenRadius == 0  Camera.hh:62-64
            V3 sample = corner + horizontal * s + vertical * t;                       // Camera.hh:66
            V3 d = normalize(sample - origin);                                        // Camera.hh:68 -> Ray ctor
            store_ray(rays[i], origin, d, FLT_MAX);
        }
    });
}

void trqh_rng_frame_begin(uint32_t* rngState, uint64_t nPixels) {      // toRNG's entry quirk: see include/tracer_rq.h
    for (uint64_t i = 0; i < nPixels; ++i) {
        uint32_t* t = rngState + 4 * i;
        std::swap(t[0], t[2]);
        std::swap(t[1], t[3]);
    }
}

uint64_t trqh_gen_bounce_rays(const trq_hit_record* recs, uint64_t n, uint64_t seedBase,
                              trq_ray* rays, uint32_t* srcIndex) {
    return trqh_gen_bounce_rays_rng(recs, n, seedBase, nullptr, nullptr, rays, srcIndex);
}

uint64_t trqh_gen_bounce_rays_rng(const trq_hit_record* recs, uint64_t n, uint64_t seedBase, const uint32_t* pixelOf,
                                  uint32_t* rngState, trq_ray* rays, uint32_t* srcIndex) {
    uint64_t k = 0;
    for (uint64_t i = 0; i < n; ++i) {
        const trq_hit_record& h = recs[i];
        if (!h.hit) continue;
        RngSlot rs(seedBase, i, pixelOf, rngState);
        Pcg32& rng = rs.rng;
        float u0 = rng.randomF(), u1 = rng.randomF();                                 // xsampler.sample2D()  Render.metal:447
        V3 p{h.p[0], h.p[1], h.p[2]}, sn{h.sn[0], h.sn[1], h.sn[2]};
        V3 origin = offset_ray(p, sn);                                                // :450
        V3 nx, ny;
        coordinate_system(sn, nx, ny);                                                // :453-455
        V3 wi = cosine_sample_hemisphere(u0, u1);                                     // Lambert S_F
        V3 dir = nx * wi.x + ny * wi.y + sn * wi.z;                                   // stw * wi  :475
        dir = normalize(dir);                                                         // ray.update -> normalize  Ray.hh:25-28
        store_ray(rays[k], origin, dir, FLT_MAX);
        if (srcIndex) srcIndex[k] = rs.pixel;
        ++k;
    }
    return k;
}

uint64_t trqh_gen_shadow_rays(const trq_hit_record* recs, uint64_t n, uint64_t seedBase,
                              const void* lightA, const void* lightB, trq_ray* rays, uint32_t* srcIndex) {
    return trqh_gen_shadow_rays_rng(recs, n, seedBase, nullptr, nullptr, lightA, lightB, rays, srcIndex);
}

uint64_t trqh_gen_shadow_rays_rng(const trq_hit_record* recs, uint64_t n, uint64_t seedBase, const uint32_t* pixelOf,
                                  uint32_t* rngState, const void* lightA, const void* lightB, trq_ray* rays, uint32_t* srcIndex) {
    const trq::RefSquare* L[2] = {(const trq::RefSquare*)lightA, (const trq::RefSquare*)lightB};
    uint64_t k = 0;
    for (uint64_t i = 0; i < n; ++i) {
        const trq_hit_record& h = recs[i];
        if (!h.hit) continue;
        RngSlot rs(seedBase, i, pixelOf, rngState);
        Pcg32& rng = rs.rng;
        float u0 = rng.randomF(), u1 = rng.randomF();                                 // Render.metal:313
        V3 p{h.p[0], h.p[1], h.p[2]}, sn{h.sn[0], h.sn[1], h.sn[2]};
        V3 origin = offset_ray(p, sn);                                                // :316
        const trq::RefSquare* sq = (rng.randomF() < 0.5f) ? L[0] : L[1];              // :319-323
        // Square::sample  Square.hh:40-58
        V3 lp{0, 0, 0};
        set(lp, sq->axis_k, sq->value_k);
        set(lp, sq->axis_i, sq->range_i[0] + u0 * (sq->range_i[1] - sq->range_i[0]));
        set(lp, sq->axis_j, sq->range_j[0] + u1 * (sq->range_j[1] - sq->range_j[0]));
        V3 ln{0, 0, 0};
        set(ln, sq->axis_k, 1.0f);
        V3 w = normalize(origin - lp);
        set(ln, sq->axis_k, copysignf(1.0f, dot(w, ln)));
        lp = offset_ray(lp, ln);
        V3 dirv = lp - origin;                                                        // Render.metal:325
        V3 nor = normalize(dirv);                                                     // :326
        float dis = length(dirv);                                                     // :334
        V3 d = normalize(nor);                                                        // Ray(_origin, _nor) normalises again  :335
        store_ray(rays[k], origin, d, dis);
        if (srcIndex) srcIndex[k] = rs.pixel;
        ++k;
    }
    return k;
}

}  // extern "C"
