// Packed fp32 arithmetic: `F2` = two fp32 values in one 64-bit register pair, processed with sm_100's packed-FP32
// instructions (PTX add/sub/mul/fma .f32x2 -> SASS FADD2 / FMUL2 / FFMA2).  The two halves hold the same quantity of two
// neighbouring DoFs (2k, 2k+1) of ONE trajectory sample, or of two neighbouring links of the sphere field
// (sgpmp_cost_pairs.cuh, the role-split fused kernel).
//
// Why: the fused kernel is bound by the single issue port of each SM sub-partition (1 warp instruction per
// clock), not by the FP32 lanes: FFMA2 performs two FMAs per lane per ISSUED instruction (it occupies the FMA
// pipe for two passes, so peak FLOP/s is unchanged — measured 70.6 TFLOP/s for both forms) and frees every
// second FP issue slot for the integer (Philox), MUFU and LDS instructions of the same warp
// (profiles/r1/ffma2_probe.txt: 128 FFMA + 64 LOP3 = 4.25 ms, 64 FFMA2 + 64 LOP3 = 3.37 ms).
// Scalars broadcast for free: ptxas turns pack(s, s) into the `R.F32` broadcast operand form, and lane extraction is
// register-pair aliasing.  The scalar overloads below (float / double) serve the one-sample-per-thread code.
#pragma once
#include "sgpmp_common.cuh"

namespace sgpmp {

struct F2 {
    unsigned long long v;
};

__device__ __forceinline__ F2 f2(float a, float b) {
    F2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r.v) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ float lane0(F2 a) { float x, y; asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(a.v)); return x; }
__device__ __forceinline__ float lane1(F2 a) { float x, y; asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(a.v)); return y; }

__device__ __forceinline__ F2 operator+(F2 a, F2 b) { F2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v)); return r; }
__device__ __forceinline__ F2 operator-(F2 a, F2 b) { F2 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v)); return r; }
__device__ __forceinline__ F2 operator*(F2 a, F2 b) { F2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v)); return r; }
__device__ __forceinline__ F2 operator+(F2 a, float s) { return a + f2(s, s); }
__device__ __forceinline__ F2 operator+(float s, F2 a) { return f2(s, s) + a; }
__device__ __forceinline__ F2 operator-(F2 a, float s) { return a - f2(s, s); }
__device__ __forceinline__ F2 operator-(float s, F2 a) { return f2(s, s) - a; }
__device__ __forceinline__ F2 operator*(F2 a, float s) { return a * f2(s, s); }
__device__ __forceinline__ F2 operator*(float s, F2 a) { return f2(s, s) * a; }
__device__ __forceinline__ F2& operator+=(F2& a, F2 b) { a = a + b; return a; }

// a * b + c in one rounding
__device__ __forceinline__ float vfma(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double vfma(double a, double b, double c) { return fma(a, b, c); }
__device__ __forceinline__ F2 vfma(F2 a, F2 b, F2 c) { F2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r.v) : "l"(a.v), "l"(b.v), "l"(c.v)); return r; }
__device__ __forceinline__ F2 vfma(float a, F2 b, F2 c) { return vfma(f2(a, a), b, c); }
__device__ __forceinline__ F2 vfma(F2 a, float b, F2 c) { return vfma(a, f2(b, b), c); }
__device__ __forceinline__ F2 vfma(F2 a, F2 b, float c) { return vfma(a, b, f2(c, c)); }
__device__ __forceinline__ F2 vfma(float a, F2 b, float c) { return vfma(f2(a, a), b, f2(c, c)); }
__device__ __forceinline__ F2 vfma(F2 a, float b, float c) { return vfma(a, f2(b, b), f2(c, c)); }

// 2^x (fp32: ex2.approx) / e^x (fp64) — the RBF kernels pre-scale their exponent accordingly
__device__ __forceinline__ float vexp2_fast(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ double vexp2_fast(double x) { return exp(x); }
__device__ __forceinline__ F2 vexp2_fast(F2 x) { return f2(vexp2_fast(lane0(x)), vexp2_fast(lane1(x))); }

// sin/cos of joint angles of the generic FK chain (fk_visit_links).  fp32: branch-free on the FMA pipe — x = j pi + r with j = rint(x / pi) (magic-number rounding,
// two-term Cody-Waite), sin x = (-1)^j sin r, cos x = (-1)^j cos r, minimax polynomials on |r| <= pi/2 (max abs error
// 1.2e-7 on |x| <= 4.5, the fp32 rounding floor of values near 1).  Reducing by pi instead of pi/2 costs two more
// polynomial terms but removes the quadrant swap: the sign is ONE xor per output with the parity bit of the magic
// sum.  fp64: libdevice.
__device__ __forceinline__ void vsincos(double x, double* s, double* c) { sincos(x, s, c); }
#define SGPMP_SIN_C0 -0.1666666716337204f
#define SGPMP_SIN_C1 0.008333331905305386f
#define SGPMP_SIN_C2 -0.00019840880122501403f
#define SGPMP_SIN_C3 2.7522235086507862e-06f
#define SGPMP_SIN_C4 -2.377893792981922e-08f
#define SGPMP_COS_C0 -0.5f
#define SGPMP_COS_C1 0.0416666604578495f
#define SGPMP_COS_C2 -0.0013888651737943292f
#define SGPMP_COS_C3 2.477461748640053e-05f
#define SGPMP_COS_C4 -2.629822404287552e-07f
__device__ __forceinline__ void vsincos(float x, float* sp, float* cp) {
    const float t = fmaf(x, 0.3183098861837907f, 12582912.0f);   // 1.5 * 2^23: rint(x / pi) lands in the low mantissa bits
    const unsigned sb = __float_as_uint(t) << 31;
    const float j = t - 12582912.0f;
    float r = fmaf(j, -3.1415927410125732f, x);        // pi = C1 + C2
    r = fmaf(j, 8.742277657347586e-08f, r);
    const float z = r * r;
    const float ps = fmaf(fmaf(fmaf(fmaf(SGPMP_SIN_C4, z, SGPMP_SIN_C3), z, SGPMP_SIN_C2), z, SGPMP_SIN_C1), z, SGPMP_SIN_C0) * z;
    const float s = fmaf(ps, r, r);
    const float c = fmaf(fmaf(fmaf(fmaf(fmaf(SGPMP_COS_C4, z, SGPMP_COS_C3), z, SGPMP_COS_C2), z, SGPMP_COS_C1), z, SGPMP_COS_C0), z, 1.0f);
    *sp = __uint_as_float(__float_as_uint(s) ^ sb);
    *cp = __uint_as_float(__float_as_uint(c) ^ sb);
}

}  // namespace sgpmp
