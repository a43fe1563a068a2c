// Counter-based normal stream of the sampler (stands in for torch's `normal_()` at
// torch/distributions/multivariate_normal.py:253; the reference's generator is not reproducible on a
// GPU, parity with it uses injected eps).  The stream definition is restated in oracle/philox.py.
//
//   Philox4x32-R, R = SGPMP_PHILOX_ROUNDS = 7 (the Crush-resistant round count of Salmon et al., SC'11, table 2;
//   R = 10 adds a safety margin that costs 12 more integer instructions per call — 6 % of the fused Panda kernel),
//   key = (seed_lo, seed_hi),
//   counter = ((t << 8) | k, sample, global particle id, draw index),   k = DoF PAIR (2k, 2k+1)
//   4 words -> two Box-Muller pairs ->   (w0, w1) -> eps[t][pos][2k], eps[t][pos][2k+1]
//                                        (w2, w3) -> eps[t][vel][2k], eps[t][vel][2k+1]
//   odd DoF count, last pair (2k+1 == n): (w0, w1) -> eps[t][pos][2k], eps[t][vel][2k];  (w2, w3) unused
//
// One call yields every normal a DoF pair needs at ONE time step, which is exactly what the dof-pair packed
// arithmetic consumes (sgpmp_cost_pairs.cuh): nothing is carried over to the next step in registers.
#pragma once
#include "sgpmp_common.cuh"
#include "sgpmp_vec.cuh"

#ifndef SGPMP_PHILOX_ROUNDS
#define SGPMP_PHILOX_ROUNDS 7
#endif

namespace sgpmp {

// The round keys k + r * (0x9E3779B9, 0xBB67AE85) are launch constants: the host precomputes them (make_rng_key) and the
// kernels read them as constant-bank operands of the LOP3s, instead of 2 R integer adds per call.
struct RngKey {
    uint32_t rk0[SGPMP_PHILOX_ROUNDS], rk1[SGPMP_PHILOX_ROUNDS];
    uint32_t draw;
};
inline RngKey make_rng_key(uint64_t seed, uint32_t draw) {
    RngKey k;
    uint32_t k0 = (uint32_t)(seed & 0xffffffffu), k1 = (uint32_t)(seed >> 32);
    for (int r = 0; r < SGPMP_PHILOX_ROUNDS; ++r) {
        k.rk0[r] = k0; k.rk1[r] = k1;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    k.draw = draw;
    return k;
}

static_assert(SGPMP_PHILOX_ROUNDS >= 3, "the factored draw (philox_prefix / philox_finish) takes rounds 0-2 apart");
constexpr uint32_t PHILOX_M0 = 0xD2511F53u, PHILOX_M1 = 0xCD9E8D57u;

__host__ __device__ __forceinline__ uint32_t philox_mulhi(uint32_t m, uint32_t a) {
#ifdef __CUDA_ARCH__
    return __umulhi(m, a);
#else
    return (uint32_t)(((uint64_t)m * a) >> 32);
#endif
}

__host__ __device__ __forceinline__ uint4 philox4x32(uint4 c, const RngKey& key) {
#pragma unroll
    for (int r = 0; r < SGPMP_PHILOX_ROUNDS; ++r) {
        const uint32_t hi0 = philox_mulhi(PHILOX_M0, c.x), lo0 = PHILOX_M0 * c.x;
        const uint32_t hi1 = philox_mulhi(PHILOX_M1, c.z), lo1 = PHILOX_M1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ key.rk0[r], lo1, hi0 ^ c.w ^ key.rk1[r], lo0);
    }
    return c;
}

// philox4x32 of the counter (x, sample, pgid, w), factored for a kernel that draws many samples of one particle and draw:
//   round 0  x1 = hi(M1 pgid) ^ sample ^ rk0[0]         per sample;   y1 = lo(M1 pgid), z1 = hi(M0 x) ^ w ^ rk1[0], w1 = lo(M0 x)
//   round 1  (hi, lo)(M0 x1) per sample;  (hi, lo)(M1 z1) uniform  ->  x2, y2 uniform;  z2 = hi(M0 x1) ^ w1 ^ rk1[1], w2 = lo(M0 x1)
//   round 2  (hi, lo)(M0 x2) uniform;  (hi, lo)(M1 z2) per sample
// philox_prefix holds the four words of rounds 0-2 that do not depend on the sample (one per (t, k) of a particle and draw),
// philox_lane the pair (hi, lo)(M0 x1) that depends on the sample and the particle only, and philox_finish the rest: 1 + 2 (R - 3)
// multiplies per call instead of 2 R.  Only XORs and exact integer products are regrouped: the words are philox4x32's.
__host__ __device__ __forceinline__ uint4 philox_prefix(uint32_t x, uint32_t pgid, uint32_t w, const RngKey& key) {
    const uint32_t y1 = PHILOX_M1 * pgid;
    const uint32_t z1 = philox_mulhi(PHILOX_M0, x) ^ w ^ key.rk1[0], w1 = PHILOX_M0 * x;
    const uint32_t x2 = philox_mulhi(PHILOX_M1, z1) ^ y1 ^ key.rk0[1], y2 = PHILOX_M1 * z1;
    return make_uint4(w1 ^ key.rk1[1], y2 ^ key.rk0[2], philox_mulhi(PHILOX_M0, x2) ^ key.rk1[2], PHILOX_M0 * x2);
}
__host__ __device__ __forceinline__ uint2 philox_lane(uint32_t sample, uint32_t pgid, const RngKey& key) {
    const uint32_t x1 = philox_mulhi(PHILOX_M1, pgid) ^ sample ^ key.rk0[0];
    return make_uint2(philox_mulhi(PHILOX_M0, x1), PHILOX_M0 * x1);
}
__host__ __device__ __forceinline__ uint4 philox_finish(uint4 u, uint2 l, const RngKey& key) {
    const uint32_t z2 = l.x ^ u.x;
    uint4 c = make_uint4(philox_mulhi(PHILOX_M1, z2) ^ u.y, PHILOX_M1 * z2, u.z ^ l.y, u.w);
#pragma unroll
    for (int r = 3; r < SGPMP_PHILOX_ROUNDS; ++r) {
        const uint32_t hi0 = philox_mulhi(PHILOX_M0, c.x), lo0 = PHILOX_M0 * c.x;
        const uint32_t hi1 = philox_mulhi(PHILOX_M1, c.z), lo1 = PHILOX_M1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ key.rk0[r], lo1, hi0 ^ c.w ^ key.rk1[r], lo0);
    }
    return c;
}
// the counter word x of time step t, DoF pair k
__host__ __device__ __forceinline__ uint32_t philox_x(uint32_t t, uint32_t k) { return (t << 8) | k; }

// u1 = (w0 + 0.5) 2^-32, u2 = (w1 + 0.5) 2^-32; r = sqrt(-2 ln u1); th = pi (2 u2 - 1)
// fp32: MUFU forms — lg2.approx (|err| <= 2^-22 abs), sqrt.approx, sin/cos.approx on [-pi, pi) (|err| <= 2^-20.9
// abs): ~12 issue slots per pair instead of ~66 for logf + sqrtf + sincospif, with |d eps| <~ 1e-6 except in the
// vanishing-radius corner u1 -> 1 (the variate stays N(0,1) to that accuracy; parity uses injected eps).
__device__ __forceinline__ void box_muller_polar(uint32_t w0, uint32_t w1, float& r, float& c, float& s) {
    const float u1 = fmaf((float)w0, 2.3283064365386963e-10f, 1.1641532182693481e-10f);
    const float th = fmaf((float)w1, 1.4629180792671596e-09f, 7.314590396335798e-10f - 3.14159265358979f);
    float l2;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l2) : "f"(u1));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-1.3862943611198906f * l2));      // -2 ln2 * log2(u1)
    asm("sin.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(th));
    asm("cos.approx.ftz.f32 %0, %1;" : "=f"(c) : "f"(th));
}
__device__ __forceinline__ void box_muller(uint32_t w0, uint32_t w1, float& z0, float& z1) {
    float r, c, s;
    box_muller_polar(w0, w1, r, c, s);
    z0 = r * c;
    z1 = r * s;
}
// both normals of one Box-Muller pair as a packed value: ONE FMUL2 (r, r) * (cos, sin)
__device__ __forceinline__ F2 box_muller2(uint32_t w0, uint32_t w1) {
    float r, c, s;
    box_muller_polar(w0, w1, r, c, s);
    return f2(c, s) * f2(r, r);
}
__device__ __forceinline__ void box_muller(uint32_t w0, uint32_t w1, double& z0, double& z1) {
    const double u1 = ((double)w0 + 0.5) * 2.3283064365386963e-10;
    const double v = ((double)w1 + 0.5) * 4.6566128730773926e-10 - 1.0;
    const double r = sqrt(-2.0 * log(u1));
    double s, c;
    sincospi(v, &s, &c);
    z0 = r * c;
    z1 = r * s;
}

// draw_offset: added to key.draw (the fused kernels run iteration `it` of a launch with draw index key.draw + it)
__device__ __forceinline__ uint4 rng_words(const RngKey& key, uint32_t t, uint32_t k, uint32_t sample, uint32_t particle_gid,
                                           uint32_t draw_offset = 0) {
    return philox4x32(make_uint4(philox_x(t, k), sample, particle_gid, key.draw + draw_offset), key);
}

// The normals of DoF pair k = (2k, 2k+1) at time step t: positions (p0, p1), velocities (v0, v1).
// full = (2k + 1 < n); the odd tail pair gets p1 = v1 = 0 (the ghost DoF of the packed kernels).
template <typename real>
__device__ __forceinline__ void normal_pair(uint4 w, bool full, real& p0, real& p1, real& v0, real& v1) {
    if (full) {
        box_muller(w.x, w.y, p0, p1);
        box_muller(w.z, w.w, v0, v1);
    } else {
        box_muller(w.x, w.y, p0, v0);
        p1 = (real)0;
        v1 = (real)0;
    }
}
template <typename real>
__device__ __forceinline__ void normal_pair(const RngKey& key, uint32_t t, uint32_t k, bool full, uint32_t sample,
                                            uint32_t particle_gid, real& p0, real& p1, real& v0, real& v1, uint32_t draw_offset = 0) {
    normal_pair<real>(rng_words(key, t, k, sample, particle_gid, draw_offset), full, p0, p1, v0, v1);
}
// packed fp32 form: ep = (eps_pos[2k], eps_pos[2k+1]), ev = (eps_vel[2k], eps_vel[2k+1])
template <bool FULL>
__device__ __forceinline__ void normal_pair_f2(uint4 w, F2& ep, F2& ev) {
    if constexpr (FULL) {
        ep = box_muller2(w.x, w.y);
        ev = box_muller2(w.z, w.w);
    } else {
        float z0, z1;
        box_muller(w.x, w.y, z0, z1);
        ep = f2(z0, 0.f);
        ev = f2(z1, 0.f);
    }
}
template <bool FULL>
__device__ __forceinline__ void normal_pair_f2(const RngKey& key, uint32_t t, uint32_t k, uint32_t sample,
                                               uint32_t particle_gid, F2& ep, F2& ev, uint32_t draw_offset = 0) {
    normal_pair_f2<FULL>(rng_words(key, t, k, sample, particle_gid, draw_offset), ep, ev);
}

}  // namespace sgpmp
