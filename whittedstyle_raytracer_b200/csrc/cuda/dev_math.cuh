// dev_math.cuh — device float3 helpers in the reference's rounding order
// (include/Vector.hpp:59-139).  The translation unit is compiled with
// -fmad=false, IEEE division and square root, no flush-to-zero, so every
// operator below is exactly one correctly-rounded float operation and the
// results equal the x86-64 (-O2, no FMA) reference bit for bit.
#pragma once
#include <cfloat>
#include <cuda_runtime.h>

namespace wrt {

struct f3 {
    float x, y, z;
};

__device__ __forceinline__ f3 mk3(float x, float y, float z) { f3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ f3 mk3(const float4& v) { return mk3(v.x, v.y, v.z); }
__device__ __forceinline__ f3 operator+(f3 a, f3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ f3 operator-(f3 a, f3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ f3 operator-(f3 a) { return mk3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ f3 operator*(f3 a, float c) { return mk3(a.x * c, a.y * c, a.z * c); }
__device__ __forceinline__ f3 operator*(float c, f3 a) { return mk3(a.x * c, a.y * c, a.z * c); }
__device__ __forceinline__ f3 operator*(f3 a, f3 b) { return mk3(a.x * b.x, a.y * b.y, a.z * b.z); }
__device__ __forceinline__ float dot(f3 a, f3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ float norm(f3 a) { return sqrtf(a.x * a.x + a.y * a.y + a.z * a.z); }
__device__ __forceinline__ f3 cross(f3 a, f3 b) {
    return mk3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ f3 normalized(f3 v) {         // Vector.hpp:127-134
    float mag = sqrtf(v.x * v.x + v.y * v.y + v.z * v.z);
    if (mag > 0) {
        float mag_inv = 1 / mag;
        return mk3(v.x * mag_inv, v.y * mag_inv, v.z * mag_inv);
    }
    return v;
}
__device__ __forceinline__ bool float_equal(float x, float y) { return fabsf(x - y) < 0.00001f; }  // global.hpp:92-94

// powf as the reference's libm computes it.  glibc's powf is correctly rounded
// in all but ~0.1 % of arguments (measured, DESIGN.md); CUDA's powf is a 4-ulp
// approximation.  x^2 is exact via one multiplication (glibc powf(x,2) == x*x
// on 2e7 samples); other exponents go through double pow and one rounding.
__device__ __forceinline__ float ref_pow2(float x) { return x * x; }
__device__ __forceinline__ float ref_powf(float x, float y) { return (float)pow((double)x, (double)y); }

__device__ __forceinline__ float4 ldg4(const float4* p) { return __ldg(p); }

// One 256-bit read-only load (sm_100: LDG.E.256) of two adjacent float4 — a whole 32-byte tree record or primitive box.
// p must be 32-byte aligned.  Divergent lanes cost the L1 one wavefront per lane and instruction, so a record fetched
// as one 256-bit load costs half the wavefronts of two 128-bit loads (the deep closest-hit levels ran the L1 data
// pipe at 82-87 % of its wavefront peak, profiles/NOTES.md).
__device__ __forceinline__ void ldg8(const float4* p, float4& a, float4& b) {
    unsigned long long q0, q1, q2, q3;
    asm("ld.global.nc.v4.b64 {%0,%1,%2,%3}, [%4];" : "=l"(q0), "=l"(q1), "=l"(q2), "=l"(q3) : "l"(p));
    a.x = __uint_as_float((unsigned)q0); a.y = __uint_as_float((unsigned)(q0 >> 32));
    a.z = __uint_as_float((unsigned)q1); a.w = __uint_as_float((unsigned)(q1 >> 32));
    b.x = __uint_as_float((unsigned)q2); b.y = __uint_as_float((unsigned)(q2 >> 32));
    b.z = __uint_as_float((unsigned)q3); b.w = __uint_as_float((unsigned)(q3 >> 32));
}

} // namespace wrt
