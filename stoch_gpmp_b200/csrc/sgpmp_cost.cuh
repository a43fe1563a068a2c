// Per-trajectory-sample cost accumulation shared by the standalone cost kernel (K3) and the fused
// iteration kernel.  One thread owns one trajectory sample and is fed its states x_t in time order.
//
// Reference being replaced (all under /root/reference/stoch_gpmp):
//   CostComposite.eval      costs/cost_functions.py:47-58  (FK hook, sum of children in list order)
//   CostGP.eval             costs/cost_functions.py:128-146 + GPFactor.get_error costs/factors/gp_factor.py:54-58
//   CostGoalPrior.eval      costs/cost_functions.py:376-388 (goal of particle p is p // K)
//   CostCollision.eval      costs/cost_functions.py:247-261 + FieldFactor costs/factors/field_factor.py:18-32
//                           (steps 1..T-1 only)
//   ObstacleMap.get_collisions   envs/obst_map.py:164-182
//   LinkDistanceField 'rbf'      costs/fields.py:63-79   (+ link interpolation :68-74)
//   CostGoal + EESE3DistanceField   costs/cost_functions.py:282-321, costs/fields.py:130-153 (last step, last link frame)
//   FK hook                      costs/cost_functions.py:51-52 (torch_robotics chain, restated from the URDF)
//   IS term                      planner.py:233-236   tau * x^T Sigma^-1 mu  ==  tau * sum_t x_t . b_t, b = P mu
#pragma once
#include <math.h>

#include "sgpmp_common.cuh"
#include "sgpmp_vec.cuh"

namespace sgpmp {

// The sphere / self RBFs evaluate exp(k d^2) as vexp2_fast(k' d^2): in fp32 k' = k log2(e) and the exponential is
// ex2.approx (2 ulp; the terms are in (0,1]); in fp64 k' = k and it is libdevice exp.

// Per-CTA constants staged in shared memory by the caller.
template <typename real>
struct CostSmem {
    const real* start;   // [d]
    const real* goal;    // [d] goal of this particle (or null)
    const real* bvec;    // [T][d]   b = Sigma^-1 mu of this particle
    const real* sph;     // [O][8]   (cx, cy, cz, k, ax, ay, az, b): k = -0.5/r^2 (* log2 e in fp32),
                         //          a = -2 k c, b = k |c|^2  so that  k |p - c|^2 = k |p|^2 + a.p + b
    const real* map;     // occupancy map of this problem (global memory)
    const uint8_t* map_u8;   // byte copy of it, or null
    real coll_const;     // RBF sum of the link frames whose position does not depend on q (structured chains)
    real self_const;     // q-independent part of the self-collision sum (structured chains)
    real mub;            // mu^T Sigma^-1 mu of this particle (fp64-accumulated): x^T b = mu^T b + (x - mu)^T b
};

constexpr int SPH_STRIDE = 8;
constexpr int SPH_ORIGIN = SPH_STRIDE * SGPMP_MAX_SPHERES + 4;     // (ox, oy, oz, -) of the shifted RBF frame, 16-byte aligned

// 4 consecutive reals from a 16-byte (fp32) / 32-byte (fp64) aligned shared-memory address in one LDS
__device__ __forceinline__ void load4(const float* p, float& a, float& b, float& c, float& d) {
    const float4 v = *reinterpret_cast<const float4*>(p);
    a = v.x; b = v.y; c = v.z; d = v.w;
}
__device__ __forceinline__ void load4(const double* p, double& a, double& b, double& c, double& d) {
    const double2 v = *reinterpret_cast<const double2*>(p), w = *reinterpret_cast<const double2*>(p + 2);
    a = v.x; b = v.y; c = w.x; d = w.y;
}

// Stage one sphere (cx, cy, cz, r) into the shared table row.
// mode != SGPMP_FIELD_RBF: slot 3 holds the radius itself (the sdf / occupancy variants need |p - c| and r).
// (ox, oy, oz): origin of the SHIFTED frame the structured chain code evaluates the RBF in (see stage_cta_constants);
// zero for every other path.
template <typename real>
__device__ __forceinline__ void stage_sphere(const real* s4, real* row, int mode, double ox = 0.0, double oy = 0.0, double oz = 0.0) {
    const double cx = (double)s4[0] - ox, cy = (double)s4[1] - oy, cz = (double)s4[2] - oz, r = s4[3];
    if (mode != SGPMP_FIELD_RBF) {
        row[0] = (real)cx; row[1] = (real)cy; row[2] = (real)cz; row[3] = (real)r;
        row[4] = row[5] = row[6] = row[7] = 0;
        return;
    }
    const double k = (sizeof(real) == 4 ? -0.5 * 1.4426950408889634 : -0.5) / (r * r);
    row[0] = (real)cx; row[1] = (real)cy; row[2] = (real)cz; row[3] = (real)k;
    row[4] = (real)(-2.0 * k * cx); row[5] = (real)(-2.0 * k * cy); row[6] = (real)(-2.0 * k * cz);
    row[7] = (real)(k * (cx * cx + cy * cy + cz * cz));
}

__device__ __forceinline__ float vsqrt(float x) { return sqrtf(x); }
__device__ __forceinline__ double vsqrt(double x) { return sqrt(x); }
__device__ __forceinline__ float vmaxv(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ double vmaxv(double a, double b) { return fmax(a, b); }
__device__ __forceinline__ float vminv(float a, float b) { return fminf(a, b); }
__device__ __forceinline__ double vminv(double a, double b) { return fmin(a, b); }
__device__ __forceinline__ float vstep_pos(float a) { return a > 0.f ? 1.f : 0.f; }        // 1 where a > 0
__device__ __forceinline__ double vstep_pos(double a) { return a > 0.0 ? 1.0 : 0.0; }
template <typename V> __device__ __forceinline__ V vneg(V a) { return -a; }
template <> __device__ __forceinline__ F2 vneg<F2>(F2 a) { return f2(-lane0(a), -lane1(a)); }   // folds into operand modifiers

// Forward kinematics of a serial arm (frames 0..N-1: fixed transform then revolute-z joint f; frames
// N..n_frames-1 fixed), calling visit(x, y, z) for every link-frame origin in chain order
// (base first if include_base).  Chain constants come from the kernel-parameter constant bank.
template <typename real, int N, typename F>
__device__ __forceinline__ void fk_visit_links(const CostParams<real>& P, const real* q, F&& visit) {
    const real one = 1, zero = 0;
    real R0 = one, R1 = zero, R2 = zero, R3 = zero, R4 = one, R5 = zero, R6 = zero, R7 = zero, R8 = one;
    real px = zero, py = zero, pz = zero;
    if (P.include_base) visit(px, py, pz);
    auto fixed = [&](int f) {
        const real* F_ = P.R[f];
        const real* tf = P.p[f];
        px = vfma(R0, tf[0], vfma(R1, tf[1], vfma(R2, tf[2], px)));
        py = vfma(R3, tf[0], vfma(R4, tf[1], vfma(R5, tf[2], py)));
        pz = vfma(R6, tf[0], vfma(R7, tf[1], vfma(R8, tf[2], pz)));
        // R <- R * F
        const real a0 = vfma(R0, F_[0], vfma(R1, F_[3], R2 * F_[6])), a1 = vfma(R0, F_[1], vfma(R1, F_[4], R2 * F_[7])), a2 = vfma(R0, F_[2], vfma(R1, F_[5], R2 * F_[8]));
        const real a3 = vfma(R3, F_[0], vfma(R4, F_[3], R5 * F_[6])), a4 = vfma(R3, F_[1], vfma(R4, F_[4], R5 * F_[7])), a5 = vfma(R3, F_[2], vfma(R4, F_[5], R5 * F_[8]));
        const real a6 = vfma(R6, F_[0], vfma(R7, F_[3], R8 * F_[6])), a7 = vfma(R6, F_[1], vfma(R7, F_[4], R8 * F_[7])), a8 = vfma(R6, F_[2], vfma(R7, F_[5], R8 * F_[8]));
        R0 = a0; R1 = a1; R2 = a2; R3 = a3; R4 = a4; R5 = a5; R6 = a6; R7 = a7; R8 = a8;
    };
#pragma unroll
    for (int f = 0; f < N; ++f) {
        fixed(f);
        // R <- R * Rz(q_f): col0' = c col0 + s col1, col1' = c col1 - s col0
        real s, c;
        vsincos(q[f], &s, &c);
        const real n0 = vfma(c, R0, s * R1), n3 = vfma(c, R3, s * R4), n6 = vfma(c, R6, s * R7);
        R1 = vfma(c, R1, vneg(s * R0)); R4 = vfma(c, R4, vneg(s * R3)); R7 = vfma(c, R7, vneg(s * R6));
        R0 = n0; R3 = n3; R6 = n6;
        visit(px, py, pz);
    }
    for (int f = N; f < P.n_frames; ++f) {   // fixed tail frames (only positions are needed downstream)
        fixed(f);
        visit(px, py, pz);
    }
}

template <typename real>
__host__ __device__ __forceinline__ bool links_interpolated(const CostParams<real>& P) {
    return (P.has_spheres && P.sphere_interp_n > 0) || (P.has_self && P.self_interp_n > 0);
}
// true when the link fields can run on the structured Panda code (CHAIN >= 1): RBF sphere field, no interpolation
template <typename real>
inline bool structured_fields_ok(const CostParams<real>& P) {
    return (P.has_spheres || P.has_self) && !links_interpolated(P) && !(P.has_spheres && P.sphere_mode != SGPMP_FIELD_RBF);
}

__device__ __forceinline__ float sg_acos(float x) { return acosf(x); }
__device__ __forceinline__ double sg_acos(double x) { return acos(x); }
__device__ __forceinline__ float sg_sqrt(float x) { return sqrtf(x); }
__device__ __forceinline__ double sg_sqrt(double x) { return sqrt(x); }
__device__ __forceinline__ void sg_sincos(float x, float* s, float* c) { sincosf(x, s, c); }
__device__ __forceinline__ void sg_sincos(double x, double* s, double* c) { sincos(x, s, c); }

// End-effector SE(3) goal cost of configuration q (CostGoal.eval cost_functions.py:308-321 over
// EESE3DistanceField.compute_cost fields.py:146-150): pose (R, p) of the LAST frame of the chain, then
//   dist = w_pos |p - p*| + w_rot acos(clamp((tr(R^T R*) - 1)/2, -1, 1));  cost = dist^2 (square) or dist.
// The weight 1/sigma_goal^2 is applied by the caller.  Runs once per trajectory sample (t = T-1), so it is kept out of
// line: the hot loop's register allocation and instruction-cache footprint do not see it.
template <typename real, int N>
__device__ __noinline__ real ee_se3_cost(const CostParams<real>& P, const real* q) {
    real R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, p[3] = {0, 0, 0};
    for (int f = 0; f < P.n_frames; ++f) {
        const real* F_ = P.R[f];
        const real* tf = P.p[f];
        real Rn[9];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            p[r] = fma(R[3 * r], tf[0], fma(R[3 * r + 1], tf[1], fma(R[3 * r + 2], tf[2], p[r])));
#pragma unroll
            for (int c = 0; c < 3; ++c)
                Rn[3 * r + c] = fma(R[3 * r], F_[c], fma(R[3 * r + 1], F_[3 + c], R[3 * r + 2] * F_[6 + c]));
        }
        if (f < N) {   // revolute z joint f: col0' = c col0 + s col1, col1' = c col1 - s col0
            real sn, cs;
            sg_sincos(q[f], &sn, &cs);
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const real a = Rn[3 * r], b = Rn[3 * r + 1];
                Rn[3 * r] = fma(cs, a, sn * b);
                Rn[3 * r + 1] = fma(cs, b, -sn * a);
            }
        }
#pragma unroll
        for (int k = 0; k < 9; ++k) R[k] = Rn[k];
    }
    const real dx = p[0] - P.ee_p[0], dy = p[1] - P.ee_p[1], dz = p[2] - P.ee_p[2];
    const real dpos = sg_sqrt(fma(dx, dx, fma(dy, dy, dz * dz)));
    real tr = 0;
#pragma unroll
    for (int k = 0; k < 9; ++k) tr = fma(R[k], P.ee_R[k], tr);
    real cs = (tr - (real)1) * (real)0.5;
    cs = cs < (real)-1 ? (real)-1 : (cs > (real)1 ? (real)1 : cs);
    const real dist = fma(P.ee_w_pos, dpos, P.ee_w_rot * sg_acos(cs));
    return P.ee_square ? dist * dist : dist;
}

// ---- structured chains ------------------------------------------------------------------------------
// CHAIN = -1: no link fields, no EE goal (planar occupancy map or no obstacle cost): the FK / field code is not compiled in at all.
// CHAIN = 0: generic serial arm (fk_visit_links, runtime constants).
// CHAIN = 1 (spheres only) / 2 (+ self-collision code): "Panda structure" (7 joints): fixed rotations are
// identity / Rx(+-90 deg) / about-z, and most translation components are zero (panda_arm_no_gripper.urdf).
// The STRUCTURE is compile-time — Rx(+-90) becomes a signed relabelling of columns, zero translation components
// vanish, the first two joints are expanded by hand — while the translation VALUES still come from the
// descriptor.  The host selects it only when the descriptor matches this structure (cos(1.57079632679) =
// 4.9e-12 is below fp32 resolution; fp64 always uses the generic path).  Further structure used: frames with
// zero translation share their parent's origin (evaluated once, weight 2); origins that do not depend on q
// (base, link1, link2) are folded into CostSmem::coll_const; joint 7 only spins the z axis along which the
// remaining translations point, so q[6] is never needed.
constexpr int PANDA_EVAL_LINKS = 6;   // link3, link4, link5(=link6), link7, link8(=hand), ee

// Joint sin/cos of the STRUCTURED Panda chain (fp32 only: standalone K3, the low-latency cost kernel, the single-role fused
// kernel): MUFU sin.approx / cos.approx, as the link warps of the role-split kernel do (sgpmp_cost_pairs.cuh) — these kernels are
// FMA-pipe bound with an idle XU pipe, and the polynomials of vsincos are ~21 FMA-pipe instructions per angle; |err| <= 2^-20.9
// displaces a link origin by < 5e-7 m (obstacle-dominated costs move by 3e-6 against the fp64 oracle, inside the 1e-5 bar).
__device__ __forceinline__ void fk_sincos(float x, float* s, float* c) { *s = __sinf(x); *c = __cosf(x); }

template <typename real>
struct Cols {   // rotation columns a, b, c
    real ax, ay, az, bx, by, bz, cx, cy, cz;
    __device__ __forceinline__ void rot_xp90() {   // R <- R Rx(+90): (a, b, c) -> (a, c, -b)
        const real tx = bx, ty = by, tz = bz;
        bx = cx; by = cy; bz = cz;
        cx = vneg(tx); cy = vneg(ty); cz = vneg(tz);
    }
    __device__ __forceinline__ void rot_xm90() {   // R <- R Rx(-90): (a, b, c) -> (a, -c, b)
        const real tx = bx, ty = by, tz = bz;
        bx = vneg(cx); by = vneg(cy); bz = vneg(cz);
        cx = tx; cy = ty; cz = tz;
    }
    __device__ __forceinline__ void rot_z(real q) {  // R <- R Rz(q): a' = c a + s b, b' = c b - s a
        real s, c;
        fk_sincos(q, &s, &c);
        rot_z_sc(s, c);
    }
    __device__ __forceinline__ void rot_z_sc(real s, real c) {
        const real nax = vfma(c, ax, s * bx), nay = vfma(c, ay, s * by), naz = vfma(c, az, s * bz);
        bx = vfma(c, bx, vneg(s * ax)); by = vfma(c, by, vneg(s * ay)); bz = vfma(c, bz, vneg(s * az));
        ax = nax; ay = nay; az = naz;
    }
};

// Origins of the 6 q-dependent, distinct link frames of the Panda structure; weights {1,1,2,1,2,1}.
// o3: origin of the shifted frame (stage_cta_constants); every origin comes out as p - o at no extra instruction.
template <typename real>
__device__ __forceinline__ void fk_panda_origins(const CostParams<real>& P, const real* q, real (&X)[PANDA_EVAL_LINKS],
                                                 real (&Y)[PANDA_EVAL_LINKS], real (&Z)[PANDA_EVAL_LINKS], const real* o3) {
    // joints 1 and 2 by hand (R starts as the identity; frame 0: t = (0,0,d1); frame 1: t = 0, Rx(-90)):
    //   a = (c1 c0, c1 s0, -s1), b = (-s1 c0, -s1 s0, -c1), c = (-s0, c0, 0),  p = (0, 0, d1)
    real s0, c0, s1, c1;
    fk_sincos(q[0], &s0, &c0);
    fk_sincos(q[1], &s1, &c1);
    const real d1 = P.p[0][2], t2y = P.p[2][1];
    const real s1c0 = s1 * c0, s1s0 = s1 * s0;
    real px = vfma(-t2y, s1c0, -o3[0]), py = vfma(-t2y, s1s0, -o3[1]), pz = vfma(-t2y, c1, d1 - o3[2]);          // frame 2: p += t2y * b
    X[0] = px; Y[0] = py; Z[0] = pz;               // link3
    // frame 2 rotation Rx(+90): (a, b, c) -> (a, c, -b)
    Cols<real> R;
    R.ax = c1 * c0; R.ay = c1 * s0; R.az = vneg(s1);
    R.bx = vneg(s0); R.by = c0; R.bz = 0;
    R.cx = s1c0; R.cy = s1s0; R.cz = c1;
    R.rot_z(q[2]);
    px = vfma(P.p[3][0], R.ax, px); py = vfma(P.p[3][0], R.ay, py); pz = vfma(P.p[3][0], R.az, pz);   // frame 3: t = (x,0,0), Rx(+90)
    X[1] = px; Y[1] = py; Z[1] = pz;               // link4
    R.rot_xp90();
    R.rot_z(q[3]);
    px = vfma(P.p[4][0], R.ax, vfma(P.p[4][1], R.bx, px));                                             // frame 4: t = (x,y,0), Rx(-90)
    py = vfma(P.p[4][0], R.ay, vfma(P.p[4][1], R.by, py));
    pz = vfma(P.p[4][0], R.az, vfma(P.p[4][1], R.bz, pz));
    X[2] = px; Y[2] = py; Z[2] = pz;               // link5 (= link6: frame 5 has t = 0)
    R.rot_xm90();
    R.rot_z(q[4]);
    R.rot_xp90();                                  // frame 5: t = 0, Rx(+90)
    R.rot_z(q[5]);
    px = vfma(P.p[6][0], R.ax, px); py = vfma(P.p[6][0], R.ay, py); pz = vfma(P.p[6][0], R.az, pz);   // frame 6: t = (x,0,0), Rx(+90)
    X[3] = px; Y[3] = py; Z[3] = pz;               // link7
    // frame 6 rotation Rx(+90) makes the new z column -b; joint 7 spins about it, so q[6] is not needed
    px = vfma(-P.p[7][2], R.bx, px); py = vfma(-P.p[7][2], R.by, py); pz = vfma(-P.p[7][2], R.bz, pz); // frame 7: t = (0,0,z)
    X[4] = px; Y[4] = py; Z[4] = pz;               // link8 (= hand: frame 8 has t = 0, rotation about z)
    px = vfma(-P.p[9][2], R.bx, px); py = vfma(-P.p[9][2], R.by, py); pz = vfma(-P.p[9][2], R.bz, pz); // frame 9: t = (0,0,z), about z
    X[5] = px; Y[5] = py; Z[5] = pz;               // ee_link
}

// Cell of position (x, y) in the occupancy map: X*(1/cell) + offset with two roundings, floor, int, clamp; value = map[iy][ix].
// The reference clamps ix with shape[0] and iy with shape[1] (obst_map.py:177-178); maps are square here.
template <typename real>
__device__ __forceinline__ int map_cell(const CostParams<real>& P, real x, real y) {
    const real xo = sg_mul_add_2r(x, P.map_inv_cell, P.map_origin_x);
    const real yo = sg_mul_add_2r(y, P.map_inv_cell, P.map_origin_y);
    int ix = (int)sg_floor(xo), iy = (int)sg_floor(yo);
    ix = min(max(ix, 0), P.map_h - 1);
    iy = min(max(iy, 0), P.map_w - 1);
    return iy * P.map_w + ix;
}

template <typename real, int N, int CHAIN = 0>
struct TrajCost {
    real c_start, c_gp, c_goal, c_coll, c_is, c_self, c_ee;
    real map_pending; // occupancy value gathered at the previous step, not yet accumulated (hides the gather latency)
    unsigned map_pending_u8;   // byte-map form of it: the RAW byte, converted when consumed
    real xp[2 * N];   // previous state

    __device__ __forceinline__ void begin() { c_start = c_gp = c_goal = c_coll = c_is = c_self = c_ee = map_pending = (real)0; map_pending_u8 = 0u; }

    // Link fields of configuration q (one FK evaluation shared by both):
    //   spheres  sum_l sum_o exp(-0.5 |p_l - c_o|^2 / r_o^2)            LinkDistanceField 'rbf'   costs/fields.py:63-79
    //   self     sum_{i,j} exp(-|p_i - p_j|^2 / (2 margin^2)), all ordered pairs incl. i == j
    //                                                                    LinkSelfDistanceField     costs/fields.py:114-124
    __device__ __forceinline__ void link_fields(const CostParams<real>& P, const CostSmem<real>& sm, const real* q) {
        const int O = P.n_spheres;
        const real zero = (real)0;
        if constexpr (CHAIN >= 1) {
            static_assert(N == 7, "Panda structure has 7 joints");
            real X[PANDA_EVAL_LINKS], Y[PANDA_EVAL_LINKS], Z[PANDA_EVAL_LINKS], PP[PANDA_EVAL_LINKS];
            fk_panda_origins(P, q, X, Y, Z, sm.sph + SPH_ORIGIN);
#pragma unroll
            for (int l = 0; l < PANDA_EVAL_LINKS; ++l) PP[l] = vfma(X[l], X[l], vfma(Y[l], Y[l], Z[l] * Z[l]));
            // (the sdf / occupancy variants of the sphere field, costs/fields.py:80-86, always take the generic chain code:
            // keeping them out of this path keeps its register footprint at that of the RBF field)
            if (P.has_spheres) {
                real acc = zero, acc2 = zero;   // acc2: links with weight 2
                for (int o = 0; o < O; ++o) {
                    const real* s = sm.sph + SPH_STRIDE * o;
                    const real k = s[3];
                    real ax, ay, az, b;
                    load4(s + 4, ax, ay, az, b);
#pragma unroll
                    for (int l = 0; l < PANDA_EVAL_LINKS; ++l) {
                        const real e = vexp2_fast(vfma(X[l], ax, vfma(Y[l], ay, vfma(Z[l], az, vfma(PP[l], k, b)))));
                        if (l == 2 || l == 4) acc2 += e; else acc += e;
                    }
                }
                c_coll += acc + (acc2 + acc2);
            }
            if (CHAIN == 2 && P.has_self) {   // CHAIN 2 = Panda structure with the self-collision code compiled in
                // weights of the 6 evaluated origins: {1,1,2,1,2,1}; constants: base (w = include_base) and
                // link1 = link2 at (0,0,z0) (w = 2).  Ordered pairs => every unordered pair counts twice.
                const real ks = P.self_k, z0 = P.p[0][2];
                real a1 = zero, a2 = zero, a4 = zero;     // sums of E over unordered pairs with weight product 1, 2, 4
#pragma unroll
                for (int l = 0; l < PANDA_EVAL_LINKS; ++l) {
                    const bool w2 = (l == 2 || l == 4);
                    const real e12 = vexp2_fast(ks * vfma((real)-2 * z0, Z[l], PP[l] + z0 * z0));    // vs link1/link2 (w = 2)
                    if (w2) a4 += e12; else a2 += e12;
                    if (P.include_base) {
                        const real eb = vexp2_fast(ks * PP[l]);                                       // vs base (w = 1)
                        if (w2) a2 += eb; else a1 += eb;
                    }
#pragma unroll
                    for (int m = l + 1; m < PANDA_EVAL_LINKS; ++m) {
                        const real dx = X[l] - X[m], dy = Y[l] - Y[m], dz = Z[l] - Z[m];
                        const real e = vexp2_fast(ks * vfma(dx, dx, vfma(dy, dy, dz * dz)));
                        const int wp = (w2 ? 2 : 1) * ((m == 2 || m == 4) ? 2 : 1);
                        if (wp == 4) a4 += e; else if (wp == 2) a2 += e; else a1 += e;
                    }
                }
                c_self += (real)2 * (a1 + ((real)2 * a2 + (real)4 * a4));
            }
        } else {
            const int mode = P.sphere_mode;
            real best = (real)-1e30;      // running max of the sdf variants over links and spheres
            auto spheres_at = [&](real x, real y, real z, real& acc) {
                for (int o = 0; o < O; ++o) {
                    const real* s = sm.sph + SPH_STRIDE * o;
                    const real dx = x - s[0], dy = y - s[1], dz = z - s[2];
                    const real d2 = vfma(dx, dx, vfma(dy, dy, dz * dz));
                    if (mode == SGPMP_FIELD_RBF) {
                        acc += vexp2_fast(s[3] * d2);
                    } else {
                        const real sd = s[3] - vsqrt(d2);
                        best = vmaxv(best, mode == SGPMP_FIELD_SDF_CLAMPED ? vminv(sd, zero) : sd);
                        acc += vstep_pos(sd);
                    }
                }
            };
            auto fold = [&](real acc) { return (mode == SGPMP_FIELD_SDF || mode == SGPMP_FIELD_SDF_CLAMPED) ? best : acc; };
            if (links_interpolated(P)) {
                // link interpolation (costs/fields.py:68-74, :117-123): keep every origin, append X_i + (X_{i+1} - X_i) alpha_k
                // for i in [lo, hi) — separately for the two fields, which carry their own (n, range)
                real PX[SGPMP_MAX_LINK_POINTS], PY[SGPMP_MAX_LINK_POINTS], PZ[SGPMP_MAX_LINK_POINTS];
                int L = 0;
                fk_visit_links<real, N>(P, q, [&](real x, real y, real z) { PX[L] = x; PY[L] = y; PZ[L] = z; ++L; });
                auto extend = [&](int n, int lo, int hi, const real* alpha) {
                    int Lx = L;
                    for (int i = lo; i < hi && n > 0; ++i)
                        for (int k = 0; k < n; ++k) {
                            PX[Lx] = PX[i] + (PX[i + 1] - PX[i]) * alpha[k];
                            PY[Lx] = PY[i] + (PY[i + 1] - PY[i]) * alpha[k];
                            PZ[Lx] = PZ[i] + (PZ[i + 1] - PZ[i]) * alpha[k];
                            ++Lx;
                        }
                    return Lx;
                };
                if (P.has_spheres) {
                    const int Lx = extend(P.sphere_interp_n, P.sphere_interp_lo, P.sphere_interp_hi, P.sphere_alpha);
                    real acc = zero;
                    for (int l = 0; l < Lx; ++l) spheres_at(PX[l], PY[l], PZ[l], acc);
                    c_coll += fold(acc);
                }
                if (P.has_self) {
                    const int Lx = extend(P.self_interp_n, P.self_interp_lo, P.self_interp_hi, P.self_alpha);
                    real sa = zero;
                    for (int l = 0; l < Lx; ++l)
                        for (int m = l + 1; m < Lx; ++m) {
                            const real dx = PX[l] - PX[m], dy = PY[l] - PY[m], dz = PZ[l] - PZ[m];
                            sa += vexp2_fast(P.self_k * vfma(dx, dx, vfma(dy, dy, dz * dz)));
                        }
                    c_self += (real)2 * sa + (real)Lx;
                }
            } else if (P.has_self) {
                // generic chain: keep every origin, then the upper triangle of the pair matrix
                real PX[SGPMP_MAX_FRAMES + 1], PY[SGPMP_MAX_FRAMES + 1], PZ[SGPMP_MAX_FRAMES + 1];
                int L = 0;
                real acc = zero;
                fk_visit_links<real, N>(P, q, [&](real x, real y, real z) {
                    PX[L] = x; PY[L] = y; PZ[L] = z; ++L;
                    if (P.has_spheres) spheres_at(x, y, z, acc);
                });
                if (P.has_spheres) c_coll += fold(acc);
                real sa = zero;
                for (int l = 0; l < L; ++l)
                    for (int m = l + 1; m < L; ++m) {
                        const real dx = PX[l] - PX[m], dy = PY[l] - PY[m], dz = PZ[l] - PZ[m];
                        sa += vexp2_fast(P.self_k * vfma(dx, dx, vfma(dy, dy, dz * dz)));
                    }
                c_self += (real)2 * sa + (real)L;
            } else {
                real acc = zero;
                fk_visit_links<real, N>(P, q, [&](real x, real y, real z) { spheres_at(x, y, z, acc); });
                c_coll += fold(acc);
            }
        }
    }

    __device__ __forceinline__ int map_index(const CostParams<real>& P, real x, real y) const { return map_cell(P, x, y); }

    // feed state x_t (t = 0..T-1 in order)
    // brow: b_t = (Sigma^-1 mu)_t of this particle (2N reals, 16-byte aligned when 2N % 4 == 0 rows are padded), or null
    // y: x - mu (the IS term is accumulated as mu^T b + y^T b: |y| << |x|, an order of magnitude less fp32 rounding)
    __device__ __forceinline__ void step(const CostParams<real>& P, const CostSmem<real>& sm, int t, int T,
                                         const real (&x)[2 * N], const real* yp, const real* yv, const real* brow) {
        if (t == 0) {
#pragma unroll
            for (int j = 0; j < 2 * N; ++j) {
                const real e = sm.start[j] - x[j];
                c_start = vfma(e, e, c_start);
            }
        } else {
#pragma unroll
            for (int i = 0; i < N; ++i) {
                const real ep = vfma(-P.dt, xp[N + i], x[i] - xp[i]);
                const real ev = x[N + i] - xp[N + i];
                c_gp = vfma(ep, vfma(P.q12x2, ev, P.q11 * ep), c_gp);
                c_gp = vfma(P.q22 * ev, ev, c_gp);
            }
            if (P.has_map) {
                // consume the gather of the PREVIOUS step, issue this step's (integer counts: exact in any order)
                if (sm.map_u8) {
                    c_coll += (real)map_pending_u8;
                    map_pending_u8 = __ldg(sm.map_u8 + map_index(P, x[0], x[1]));
                } else {
                    c_coll += map_pending;
                    map_pending = __ldg(sm.map + map_index(P, x[0], x[1]));
                }
            }
            if constexpr (CHAIN >= 0) {        // CHAIN -1: no link fields and no EE goal are compiled in (state-only costs)
                if (P.has_spheres || P.has_self) link_fields(P, sm, x);
            }
        }
        if (t == T - 1 && P.has_goal) {
#pragma unroll
            for (int j = 0; j < 2 * N; ++j) {
                const real e = sm.goal[j] - x[j];
                c_goal = vfma(e, e, c_goal);
            }
        }
        if (brow) {
            constexpr int DP4 = (2 * N + 3) / 4;
            real b[4 * DP4];
#pragma unroll
            for (int k = 0; k < DP4; ++k) load4(brow + 4 * k, b[4 * k], b[4 * k + 1], b[4 * k + 2], b[4 * k + 3]);
#pragma unroll
            for (int i = 0; i < N; ++i) c_is = vfma(yp[i], b[i], vfma(yv[i], b[N + i], c_is));
        }
#pragma unroll
        for (int j = 0; j < 2 * N; ++j) xp[j] = x[j];
    }

    __device__ __forceinline__ void finish(const CostParams<real>& P, const CostSmem<real>& sm, int T) {
        if (P.has_map) {
            c_coll += map_pending;
            c_coll += (real)map_pending_u8;
        }
        c_start = c_start * P.inv_sig_start2;
        c_goal = c_goal * P.inv_sig_goal2;
        if (CHAIN >= 1) {
            c_coll = c_coll + (real)(T - 1) * sm.coll_const;
            c_self = c_self + (real)(T - 1) * sm.self_const;
        }
        c_coll = c_coll * (P.has_map ? P.map_w_coll : P.sphere_w_coll);
        c_self = c_self * P.self_w_coll;
        c_is = (c_is + sm.mub) * P.temperature;
        // EE SE(3) goal on the last state (xp holds x_{T-1} after the final step)
        if constexpr (CHAIN >= 0) {
            if (P.has_ee) {
                real q[N];      // a COPY: taking the address of xp itself would demote the whole previous-state array to local memory
#pragma unroll
                for (int i = 0; i < N; ++i) q[i] = xp[i];
                c_ee = ee_se3_cost<real, N>(P, q) * P.ee_w;
            }
        }
    }
    // Contribution of ONE time step to the total (everything above is linear in the per-step accumulators): used by the
    // low-latency cost kernel, where a trajectory's time steps are spread over threads.  Call after begin() + step(t) on a fresh
    // object (xp preset to x_{t-1}); the q-independent constants and mu^T b are added by the thread that owns t = T-1.
    __device__ __forceinline__ real partial(const CostParams<real>& P, const CostSmem<real>& sm, int T, int t) const {
        real coll = c_coll + map_pending, self = c_self, is = c_is;
        coll = coll + (real)map_pending_u8;
        if (t == T - 1) {
            if (CHAIN >= 1) {
                coll = coll + (real)(T - 1) * sm.coll_const;
                self = self + (real)(T - 1) * sm.self_const;
            }
            is = is + sm.mub;
        }
        return ((((c_start * P.inv_sig_start2 + c_gp) + c_goal * P.inv_sig_goal2) + self * P.self_w_coll) +
                coll * (P.has_map ? P.map_w_coll : P.sphere_w_coll)) + is * P.temperature;
    }
    // summation order of the shipped examples' cost lists: CostGP (start + gp), CostGoalPrior, self-collision,
    // obstacle collision, EE goal (examples/panda_environment.py:90), then += IS (planner.py:236)
    __device__ __forceinline__ real total() const { return (((((c_start + c_gp) + c_goal) + c_self) + c_coll) + c_ee) + c_is; }
};

// Per-CTA staging of the problem constants into shared memory: start [d], goal [d] of goal index g, the sphere
// table [MAX_SPHERES][8] followed by one slot for coll_const.  Ends with a __syncthreads().
constexpr int SPH_SMEM = SPH_STRIDE * SGPMP_MAX_SPHERES + 8;   // + coll_const, self_const, -, -, origin[3], -  (keeps what follows 16-byte aligned)

// VOFF: offset of the velocity half inside the staged start/goal rows (N = dense; the dof-pair kernels pad it).
template <typename real, int N, int CHAIN, int VOFF = N>
__device__ __forceinline__ void stage_cta_constants(const CostParams<real>& P, int b, int g, int G, real* start, real* goal,
                                                    real* sph) {
    constexpr int d = 2 * N;
    for (int k = threadIdx.x; k < 2 * VOFF; k += blockDim.x) { start[k] = 0; goal[k] = 0; }
    __syncthreads();
    for (int k = threadIdx.x; k < d; k += blockDim.x) {
        const int c = k < N ? k : VOFF + (k - N);
        start[c] = P.start[(size_t)b * d + k];
        goal[c] = P.has_goal ? P.goals[((size_t)b * G + g) * d + k] : (real)0;
    }
    // Structured chains evaluate k |p - c|^2 in the EXPANDED form k |p|^2 + a.p + b (4 FMA per link-sphere pair).  Its terms are
    // ~k |c|^2 each and cancel down to k d^2, so in fp32 the exponent carries ~|k| |c|^2 2^-23 of rounding (3e-5 of the term with the
    // shipped scene seen from the robot base).  The cure costs nothing per sample: a frame whose origin is the centroid of the spheres
    // — where the exponentials that matter live — makes |c| and |p| there a few sphere radii; the origin is folded into the first
    // link offset of the chain (fk_panda_origins), so every link origin comes out already shifted.  (The self-collision code of
    // CHAIN 2 uses base-frame expressions for the q-independent links: no shift there.)
    if (threadIdx.x == 0) {
        double ox = 0, oy = 0, oz = 0;
        if (CHAIN == 1 && P.has_spheres && !P.has_self && P.sphere_mode == SGPMP_FIELD_RBF && P.n_spheres > 0) {
            const real* s4 = P.spheres + (size_t)(P.spheres_per_problem ? b : 0) * P.n_spheres * 4;
            for (int k = 0; k < P.n_spheres; ++k) { ox += s4[4 * k]; oy += s4[4 * k + 1]; oz += s4[4 * k + 2]; }
            ox /= P.n_spheres; oy /= P.n_spheres; oz /= P.n_spheres;
        }
        sph[SPH_ORIGIN] = (real)ox; sph[SPH_ORIGIN + 1] = (real)oy; sph[SPH_ORIGIN + 2] = (real)oz; sph[SPH_ORIGIN + 3] = 0;
    }
    __syncthreads();
    const double ox = sph[SPH_ORIGIN], oy = sph[SPH_ORIGIN + 1], oz = sph[SPH_ORIGIN + 2];     // the ROUNDED origin is the one the chain subtracts
    if (P.has_spheres)
        for (int k = threadIdx.x; k < P.n_spheres; k += blockDim.x)
            stage_sphere<real>(P.spheres + ((size_t)(P.spheres_per_problem ? b : 0) * P.n_spheres + k) * 4, sph + SPH_STRIDE * k, P.sphere_mode,
                               ox, oy, oz);
    __syncthreads();
    if (threadIdx.x == 0) {
        real cc = 0;
        if (CHAIN >= 1 && P.has_spheres && P.sphere_mode == SGPMP_FIELD_RBF) {
            // q-independent origins of the Panda structure: base (if counted), link1 and link2 at (0, 0, z0), in the shifted frame
            const real z0 = P.p[0][2];
            const real bx = (real)-ox, by = (real)-oy, bz = (real)-oz, lz = z0 - (real)oz;
            for (int o = 0; o < P.n_spheres; ++o) {
                const real* s = sph + SPH_STRIDE * o;
                if (P.include_base) cc += vexp2_fast(s[3] * (bx * bx + by * by + bz * bz) + (s[4] * bx + s[5] * by + s[6] * bz) + s[7]);
                cc += (real)2 * vexp2_fast(s[3] * (bx * bx + by * by + lz * lz) + (s[4] * bx + s[5] * by + s[6] * lz) + s[7]);
            }
        }
        sph[SPH_STRIDE * SGPMP_MAX_SPHERES] = cc;
        real sc = 0;
        if (CHAIN >= 1 && P.has_self) {
            // constant-constant pairs + the diagonal of the 6 evaluated origins (weights 1,1,2,1,2,1 -> 12)
            const real z0 = P.p[0][2], wb = P.include_base ? (real)1 : (real)0;
            sc = wb * wb + (real)4 + (real)4 * wb * vexp2_fast(P.self_k * z0 * z0) + (real)12;
        }
        sph[SPH_STRIDE * SGPMP_MAX_SPHERES + 1] = sc;
    }
    __syncthreads();
}

// 1 if the descriptor's chain has the Panda STRUCTURE (see fk_panda_origins); host-side check.
inline int chain_is_panda_structure(const sgpmp_cost_desc_t& d, int n_dof) {
    if (n_dof != 7 || d.n_frames != 10) return 0;
    static const int rot[10] = {0, -1, 1, 1, -1, 1, 1, 0, 2, 2};          // 0: I, +-1: Rx(+-90), 2: about z
    static const int tmask[10] = {4, 0, 2, 1, 3, 0, 1, 4, 0, 4};          // bit0 x, bit1 y, bit2 z may be non-zero
    const double tol = 1e-9;
    for (int f = 0; f < 10; ++f) {
        const double* R = d.chain_R[f];
        for (int k = 0; k < 3; ++k)
            if (!((tmask[f] >> k) & 1) && d.chain_p[f][k] != 0.0) return 0;
        double want[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
        if (rot[f] == 1) { double w[9] = {1, 0, 0, 0, 0, -1, 0, 1, 0}; memcpy(want, w, sizeof(w)); }
        if (rot[f] == -1) { double w[9] = {1, 0, 0, 0, 0, 1, 0, -1, 0}; memcpy(want, w, sizeof(w)); }
        if (rot[f] == 2) {   // rotation about z: third row/column are e_z
            if (fabs(R[2]) > tol || fabs(R[5]) > tol || fabs(R[6]) > tol || fabs(R[7]) > tol || fabs(R[8] - 1) > tol) return 0;
            continue;
        }
        for (int k = 0; k < 9; ++k)
            if (fabs(R[k] - want[k]) > tol) return 0;
    }
    return 1;
}

// Block-wide sum of one double per thread (shuffles + one shared-memory hop); scratch: >= 32 doubles.
__device__ __forceinline__ double block_sum_f64(double v, double* scratch) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (l == 0) scratch[w] = v;
    __syncthreads();
    double r = 0;
    for (int k = 0; k < nw; ++k) r += scratch[k];
    __syncthreads();
    return r;
}

// b = P mu for one particle, computed in fp64 from the D/O blocks (the fp32 reference evaluates this
// contraction with catastrophic cancellation; see DESIGN.md §5), stored as `real`.
// tabDO: [T][7] doubles (d11,d12,d22,o11,o12,o21,o22), O_t = P[t+1,t].
// MU_STRIDE: row stride of mu in reals (0 = dense rows of 2n); VOFF: offset of the velocity half (0 = n).
template <typename real, int MU_STRIDE = 0, int VOFF = 0>
__device__ __forceinline__ double precision_times_row(const double* tabDO, const real* mu, int T, int n_, int t, int i,
                                                      real* bp, real* bv) {
    const int d = MU_STRIDE ? MU_STRIDE : 2 * n_;
    const int n = VOFF ? VOFF : n_;
    const double* r = tabDO + t * 7;
    const double mp = mu[t * d + i], mv = mu[t * d + n + i];
    double p = r[0] * mp + r[1] * mv;
    double v = r[1] * mp + r[2] * mv;
    if (t > 0) {
        const double* q = tabDO + (t - 1) * 7;
        const double ap = mu[(t - 1) * d + i], av = mu[(t - 1) * d + n + i];
        p += q[3] * ap + q[4] * av;
        v += q[5] * ap + q[6] * av;
    }
    if (t < T - 1) {
        const double ap = mu[(t + 1) * d + i], av = mu[(t + 1) * d + n + i];
        p += r[3] * ap + r[5] * av;   // O_t^T
        v += r[4] * ap + r[6] * av;
    }
    *bp = (real)p;
    *bv = (real)v;
    return mp * p + mv * v;        // this row's share of mu^T P mu, in fp64
}

}  // namespace sgpmp
