// tracer_b200/csrc/kernels/producers.cuh -- device-side ray PRODUCERS (SURVEY.md section 8, row f-3).
//
// The callers either side of the ray query, so that a multi-bounce wavefront never leaves the GPU:
//   cast_rays_kernel      castRay for every pixel             Camera.hh:59-69, Render.metal:523-527 (camera from MakeCamera, Tracer.mm:87-125)
//   spawn_bounce_kernel   diffuse bounce from a hit           Render.metal:447-475 (offset_ray Math.hh:62-74, CoordinateSystem /
//                                                             CosineSampleHemisphere Sampling.hh:18-34,79-99,125-129, Ray::update Ray.hh:25-28)
//   spawn_shadow_kernel   NEE shadow ray toward a light square  Render.metal:313-337, Square::sample Square.hh:40-58
// Surviving rays are compacted into the output queue with ONE atomicAdd per warp (ballot + popc ranks);
// srcIndex[k] says which input ray (pixel) output ray k descends from. The arithmetic is the host harness's
// (csrc/host/harness.cpp), same order, strict fp32; only cosf/sinf differ from libm by ulps.
#pragma once
#include "intersect.cuh"
#include "scene_dev.cuh"
#include "../../../include/tracer_rq.h"

namespace trq {

struct CameraDev {           // struct Camera (Camera.hh:7-22), the fields castRay reads
    float lookFrom[3], u[3], v[3];
    float vertical[3], horizontal[3], corner[3];
    float lenRadius;
};

// Random.metal:3-25 (= pcg_basic.c:44-67)
struct Pcg32Dev {
    uint64_t state, inc;
    __device__ __forceinline__ Pcg32Dev(uint64_t initstate, uint64_t initseq) {
        state = 0u; inc = (initseq << 1u) | 1u;
        next(); state += initstate; next();
    }
    __device__ __forceinline__ uint32_t next() {
        const uint64_t old = state;
        state = old * 6364136223846793005ULL + inc;
        const uint32_t xorshifted = (uint32_t)(((old >> 18u) ^ old) >> 27u);
        const uint32_t rot = (uint32_t)(old >> 59u);
        return (xorshifted >> rot) | (xorshifted << ((0u - rot) & 31u));
    }
    __device__ __forceinline__ float randomF() { return fmul(__uint2float_rn(next()), 2.3283064365386963e-10f); }   // ldexp(float(i), -32)
    // the reference's per-pixel state texture (RGBA32Uint) in exRNG's layout (Render.hh:109-120):
    // {state >> 32, state, inc >> 32, inc}, on load AND store (see rng_frame_begin_kernel for toRNG's entry quirk)
    __device__ __forceinline__ void load(const uint4 t) { state = ((uint64_t)t.x << 32) | t.y; inc = ((uint64_t)t.z << 32) | t.w; }
    __device__ __forceinline__ uint4 store() const { return make_uint4((uint32_t)(state >> 32), (uint32_t)state, (uint32_t)(inc >> 32), (uint32_t)inc); }
};

// Where the draws of record i come from: the pixel's stream in the state texture (loaded here, stored back by
// rng_release) or, without a texture, PCG32(seedBase + i, 1).
__device__ __forceinline__ Pcg32Dev rng_acquire(uint64_t seedBase, uint64_t i, const uint32_t* __restrict__ pixelOf,
                                                const uint32_t* rngState, uint32_t& pixel) {
    pixel = pixelOf ? __ldg(pixelOf + i) : (uint32_t)i;
    Pcg32Dev rng(seedBase + i, 1);
    if (rngState) rng.load(*reinterpret_cast<const uint4*>(rngState + 4 * (size_t)pixel));
    return rng;
}
__device__ __forceinline__ void rng_release(const Pcg32Dev& rng, uint32_t* rngState, uint32_t pixel) {
    if (rngState) *reinterpret_cast<uint4*>(rngState + 4 * (size_t)pixel) = rng.store();
}

// Math.hh:57-74. of_i = int(256 n) with the host's conversion (host_f2i: NaN and |256 n| >= 2^31 give INT32_MIN); the
// negation and the add into the float's bits wrap modulo 2^32, as on the host.
__device__ __forceinline__ float offset_component(float p, float n) {
    const float origin = 1.0f / 32.0f, float_scale = 1.0f / 65536.0f, int_scale = 256.0f;
    const uint32_t of_i = (uint32_t)host_f2i(fmul(int_scale, n));
    const float p_i = __uint_as_float(__float_as_uint(p) + ((p < 0.0f) ? 0u - of_i : of_i));
    return fabsf(p) < origin ? fadd(p, fmul(float_scale, n)) : p_i;
}
__device__ __forceinline__ f3 offset_ray_dev(const f3& p, const f3& n) {
    return make_f3(offset_component(p.x, n.x), offset_component(p.y, n.y), offset_component(p.z, n.z));
}

// Sampling.hh:18-34
__device__ __forceinline__ void coordinate_system_dev(const f3& a, f3& b, f3& c) {
    if (fabsf(a.x) > fabsf(a.y)) b = make_f3(-a.z, 0.0f, a.x);
    else                         b = make_f3(0.0f, a.z, -a.y);
    b = normalize3(b);
    c = cross3(a, b);
}

// Sampling.hh:79-99,125-129
__device__ __forceinline__ f3 cosine_sample_hemisphere_dev(float u0, float u1) {
    const float ox = fsub(fmul(2.0f, u0), 1.0f), oy = fsub(fmul(2.0f, u1), 1.0f);
    float dx = 0.0f, dy = 0.0f;
    if (!(ox == 0.0f && oy == 0.0f)) {
        const float PiOver2 = TRQ_PI_F / 2.0f, PiOver4 = TRQ_PI_F / 4.0f;
        float theta, r;
        if (fabsf(ox) > fabsf(oy)) { r = ox; theta = fmul(PiOver4, fdiv(oy, ox)); }
        else                       { r = oy; theta = fsub(PiOver2, fmul(PiOver4, fdiv(ox, oy))); }
        dx = fmul(r, cosf(theta)); dy = fmul(r, sinf(theta));
    }
    const float z = fsqrt(fmaxf(0.0f, fsub(fsub(1.0f, fmul(dx, dx)), fmul(dy, dy))));
    return make_f3(dx, dy, z);
}

__device__ __forceinline__ void write_ray(trq_ray* out, uint64_t k, const f3& o, const f3& d, float tmax) {
    float4* p = reinterpret_cast<float4*>(out + k);
    p[0] = make_float4(o.x, o.y, o.z, tmax);
    p[1] = make_float4(d.x, d.y, d.z, 0.0f);
}

// HitRecord p / sn of a trq_hit (what the integrators read before spawning): same code as trq_expand_hits.
__device__ __forceinline__ bool surface_of_hit(const SceneDev& S, const trq_ray* __restrict__ rays, const trq_hit* __restrict__ hits,
                                               uint64_t i, Surface& s) {
    const float4 h0 = __ldg(reinterpret_cast<const float4*>(hits + i));
    const float4 h1 = __ldg(reinterpret_cast<const float4*>(hits + i) + 1);
    if ((__float_as_uint(h1.w) & TRQ_HIT_FLAG_HIT) == 0u) return false;
    const float4 r0 = __ldg(reinterpret_cast<const float4*>(rays + i));
    const float4 r1 = __ldg(reinterpret_cast<const float4*>(rays + i) + 1);
    const RayCtx ray = make_ray_ctx(r0.x, r0.y, r0.z, r1.x, r1.y, r1.z);
    const uint32_t pType = __float_as_uint(h0.y), pIndex = __float_as_uint(h0.z);
    s.p = s.gn = s.sn = make_f3(0.f, 0.f, 0.f); s.uvx = s.uvy = 0.0f; s.front = 0; s.material = 0;
    float t;
    if (pType == TRQ_TRIANGLE)     tri_surface(S.verts, S.idx, pIndex, h1.x, h1.y, ray, s);
    else if (pType == TRQ_SPHERE)  sphere_surface(&S.spheres[pIndex], h0.x, ray, s);
    else if (pType == TRQ_SQUARE)  square_hit(&S.squares[pIndex], ray, h0.x, h0.x, t, &s);
    else if (pType == TRQ_CUBE)    cube_surface(&S.cubes[pIndex], ray, h0.x, h1.x, h1.y, s);
    return true;
}

// Queue push with one atomic per warp: every lane of the warp must call it.
__device__ __forceinline__ uint64_t warp_push(bool alive, unsigned long long* counter) {
    const unsigned lane = threadIdx.x & 31u;
    const unsigned m = __ballot_sync(0xffffffffu, alive);
    unsigned long long base = 0;
    if (m != 0u && lane == (unsigned)(__ffs(m) - 1)) base = atomicAdd(counter, (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, m ? (__ffs(m) - 1) : 0);
    return base + (uint64_t)__popc(m & ((1u << lane) - 1u));
}

// toRNG at kernel entry (Render.hh:96-107, Render.metal:511-521) brace-initialises pcg32_t {state, inc} (Random.hh:6-12)
// with (inc, state): the words exRNG stored as state come back as inc and vice versa. Applying that once per frame --
// swapping the two halves of every texel -- and then using exRNG's layout for every wave reproduces the reference's
// texture from frame to frame.
__global__ void __launch_bounds__(256)
rng_frame_begin_kernel(uint4* __restrict__ rngState, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint4 t = rngState[i];
    rngState[i] = make_uint4(t.z, t.w, t.x, t.y);
}

__global__ void __launch_bounds__(256)
cast_rays_kernel(CameraDev cam, uint32_t W, uint32_t H, trq_ray* __restrict__ rays) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (uint64_t)W * H) return;
    const uint32_t x = (uint32_t)(i % W), y = (uint32_t)(i / W);
    const float s = fdiv((float)x, (float)W), t = fdiv((float)y, (float)H);            // Render.metal:523-524
    const f3 origin = ld3(cam.lookFrom);                                                // lenRadius == 0 (aperture 0)  Camera.hh:62-64
    const f3 sample = add3(add3(ld3(cam.corner), scale3(ld3(cam.horizontal), s)), scale3(ld3(cam.vertical), t));   // :66
    const f3 d = normalize3(sub3(sample, origin));                                      // :68 -> Ray ctor (Ray.hh:21-23)
    write_ray(rays, i, origin, d, FLT_MAX);
}

__global__ void __launch_bounds__(256)
spawn_bounce_kernel(SceneDev S, const trq_ray* __restrict__ rays, const trq_hit* __restrict__ hits, uint64_t n,
                    const unsigned long long* __restrict__ nPtr, uint64_t seedBase, const uint32_t* __restrict__ pixelOf,
                    uint32_t* rngState, trq_ray* __restrict__ out, uint32_t* __restrict__ srcIndex, unsigned long long* counter) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    Surface s;
    const bool alive = i < live_count(n, nPtr) && surface_of_hit(S, rays, hits, i, s);
    f3 origin = make_f3(0.f, 0.f, 0.f), dir = make_f3(0.f, 0.f, 1.f);
    uint32_t pixel = 0;
    if (alive) {
        Pcg32Dev rng = rng_acquire(seedBase, i, pixelOf, rngState, pixel);
        const float u0 = rng.randomF(), u1 = rng.randomF();                             // xsampler.sample2D()  Render.metal:447
        rng_release(rng, rngState, pixel);
        origin = offset_ray_dev(s.p, s.sn);                                             // :450
        f3 nx, ny;
        coordinate_system_dev(s.sn, nx, ny);                                            // :453-455
        const f3 wi = cosine_sample_hemisphere_dev(u0, u1);                             // Lambert S_F (MatteBXDF.hh:16-21)
        dir = add3(add3(scale3(nx, wi.x), scale3(ny, wi.y)), scale3(s.sn, wi.z));       // stw * wi  :475
        dir = normalize3(dir);                                                          // ray.update  Ray.hh:25-28
    }
    const uint64_t k = warp_push(alive, counter);
    if (alive) {
        write_ray(out, k, origin, dir, FLT_MAX);
        if (srcIndex) srcIndex[k] = pixel;
    }
}

__global__ void __launch_bounds__(256)
spawn_shadow_kernel(SceneDev S, const trq_ray* __restrict__ rays, const trq_hit* __restrict__ hits, uint64_t n,
                    const unsigned long long* __restrict__ nPtr, uint64_t seedBase, const uint32_t* __restrict__ pixelOf,
                    uint32_t* rngState, uint32_t lightA, uint32_t lightB, trq_ray* __restrict__ out,
                    uint32_t* __restrict__ srcIndex, unsigned long long* counter) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    Surface s;
    const bool alive = i < live_count(n, nPtr) && surface_of_hit(S, rays, hits, i, s);
    f3 origin = make_f3(0.f, 0.f, 0.f), dir = make_f3(0.f, 0.f, 1.f);
    float dis = 0.0f;
    uint32_t pixel = 0;
    if (alive) {
        Pcg32Dev rng = rng_acquire(seedBase, i, pixelOf, rngState, pixel);
        const float u0 = rng.randomF(), u1 = rng.randomF();                             // Render.metal:313
        origin = offset_ray_dev(s.p, s.sn);                                             // :316
        const RefSquare* sq = &S.squares[(rng.randomF() < 0.5f) ? lightA : lightB];     // :319-323
        rng_release(rng, rngState, pixel);
        // Square::sample  Square.hh:40-58
        f3 lp = make_f3(0.f, 0.f, 0.f);
        set3(lp, sq->axis_k, sq->value_k);
        set3(lp, sq->axis_i, fadd(sq->range_i[0], fmul(u0, fsub(sq->range_i[1], sq->range_i[0]))));
        set3(lp, sq->axis_j, fadd(sq->range_j[0], fmul(u1, fsub(sq->range_j[1], sq->range_j[0]))));
        f3 ln = make_f3(0.f, 0.f, 0.f);
        set3(ln, sq->axis_k, 1.0f);
        const f3 w = normalize3(sub3(origin, lp));
        set3(ln, sq->axis_k, copysignf(1.0f, dot3(w, ln)));
        lp = offset_ray_dev(lp, ln);
        const f3 dirv = sub3(lp, origin);                                               // Render.metal:325
        const f3 nor = normalize3(dirv);                                                // :326
        dis = fsqrt(dot3(dirv, dirv));                                                  // :334 length(_dir)
        dir = normalize3(nor);                                                          // Ray(_origin, _nor) normalises again  :335
    }
    const uint64_t k = warp_push(alive, counter);
    if (alive) {
        write_ray(out, k, origin, dir, dis);
        if (srcIndex) srcIndex[k] = pixel;
    }
}

}  // namespace trq
