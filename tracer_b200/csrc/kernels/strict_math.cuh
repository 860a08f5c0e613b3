// tracer_b200/csrc/kernels/strict_math.cuh
//
// fp32 arithmetic with the reference's operation ORDER and one IEEE rounding per operation.
// Every add / mul / div / sqrt goes through a round-to-nearest intrinsic, which nvcc never
// contracts into FMA, so results are bit-identical to the host oracle (g++ -ffp-contract=off)
// regardless of -fmad. Conventions (oracle/shim/metal_stdlib, SURVEY.md appendix B):
//   dot(a,b)   = (a.x*b.x + a.y*b.y) + a.z*b.z
//   cross(a,b) = (a.y*b.z - a.z*b.y, a.z*b.x - a.x*b.z, a.x*b.y - a.y*b.x)
//   normalize  = v / sqrt(dot(v,v))          min/max = fminf/fmaxf
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace trq {

struct f3 { float x, y, z; };

__device__ __forceinline__ float fadd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fsub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float fmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fdiv(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ float fsqrt(float a) { return __fsqrt_rn(a); }

// (int32_t)v as the host computes it (x86 cvttss2si): truncation toward zero, and INT32_MIN for NaN and for values outside
// [-2^31, 2^31). CUDA's (int)v saturates instead and maps NaN to 0, so offset_ray would move a point the host does not.
__device__ __forceinline__ int32_t host_f2i(float v) {
    return (v != v || v >= 0x1p31f || v < -0x1p31f) ? INT32_MIN : __float2int_rz(v);
}

__device__ __forceinline__ f3 make_f3(float x, float y, float z) { f3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ f3 ld3(const float* p) { return make_f3(p[0], p[1], p[2]); }
__device__ __forceinline__ f3 add3(f3 a, f3 b) { return make_f3(fadd(a.x, b.x), fadd(a.y, b.y), fadd(a.z, b.z)); }
__device__ __forceinline__ f3 sub3(f3 a, f3 b) { return make_f3(fsub(a.x, b.x), fsub(a.y, b.y), fsub(a.z, b.z)); }
__device__ __forceinline__ f3 mul3(f3 a, f3 b) { return make_f3(fmul(a.x, b.x), fmul(a.y, b.y), fmul(a.z, b.z)); }
__device__ __forceinline__ f3 scale3(f3 a, float s) { return make_f3(fmul(a.x, s), fmul(a.y, s), fmul(a.z, s)); }
__device__ __forceinline__ f3 divs3(f3 a, float s) { return make_f3(fdiv(a.x, s), fdiv(a.y, s), fdiv(a.z, s)); }
__device__ __forceinline__ f3 neg3(f3 a) { return make_f3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ float dot3(f3 a, f3 b) { return fadd(fadd(fmul(a.x, b.x), fmul(a.y, b.y)), fmul(a.z, b.z)); }
__device__ __forceinline__ f3 cross3(f3 a, f3 b) {
    return make_f3(fsub(fmul(a.y, b.z), fmul(a.z, b.y)),
                   fsub(fmul(a.z, b.x), fmul(a.x, b.z)),
                   fsub(fmul(a.x, b.y), fmul(a.y, b.x)));
}
__device__ __forceinline__ f3 normalize3(f3 a) { return divs3(a, fsqrt(dot3(a, a))); }
__device__ __forceinline__ float get3(f3 a, unsigned i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }
__device__ __forceinline__ void set3(f3& a, unsigned i, float v) { if (i == 0) a.x = v; else if (i == 1) a.y = v; else a.z = v; }

}  // namespace trq
