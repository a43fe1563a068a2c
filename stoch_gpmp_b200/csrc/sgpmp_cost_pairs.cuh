// fp32 cost accumulation with packed-FP32 arithmetic ACROSS THE DoFs OF ONE SAMPLE ("dof-pair" packing).
//
// Same arithmetic and reference citations as sgpmp_cost.cuh (TrajCost); what changes is the instruction
// selection.  The fused kernel is bound by the one-instruction-per-clock issue port of each SM sub-partition,
// and sm_100's FFMA2/FADD2/FMUL2 perform two fp32 operations per lane per issued instruction (sgpmp_vec.cuh).
// Here the two halves of a packed register hold the SAME quantity of two neighbouring DoFs (2k, 2k+1) of one
// trajectory sample — positions, velocities, normals, recurrence state, GP errors — or of two neighbouring
// LINKS in the sphere field.  No per-thread state is duplicated (unlike two samples per thread), so register
// use and occupancy stay those of the scalar kernel while the FP32 instruction count drops by ~45 %.
//
// Odd DoF counts are padded with a ghost DoF whose mean, normals, start/goal entries and b entries are zero:
// it contributes exactly 0 to every quadratic form.  Shared-memory rows use the layout
// [pos 0..2*NP2-1][vel 0..2*NP2-1] (NP2 = ceil(N/2)) so that every pair is one aligned 8-byte half of an LDS.128.
#pragma once
#include "sgpmp_cost.cuh"

namespace sgpmp {

// Joint sin/cos of the packed link-field code: MUFU sin.approx / cos.approx for all three joint pairs.  After the role split the
// link warps are FMA-pipe bound (132 of their 305 instructions per step are packed FP32 holding the pipe for two passes) while the
// XU pipe idled more than half of the time, and packed FMA-pipe sin/cos polynomials were 96 of those FMA cycles.  MUFU's
// |err| <= 2^-20.9 displaces a link origin by < 5e-7 m; measured where the obstacle term IS the cost
// (test_fused_link_field_term_dominating, C3 shape, fp32 vs the fp64 oracle): 9.0e-7 / 3.1e-6 with MUFU against 1.9e-7 / 3.3e-6
// with the polynomials — inside the 1e-5 bar either way.  C4: 14.59 -> 13.38 ms.
__device__ __forceinline__ void link_sincos(F2 x, F2* s, F2* c) {
    *s = f2(__sinf(lane0(x)), __sinf(lane1(x)));
    *c = f2(__cosf(lane0(x)), __cosf(lane1(x)));
}

__device__ __forceinline__ float hsum(F2 a) { return lane0(a) + lane1(a); }

template <int N, int CHAIN>
struct TrajCostPairs {
    static constexpr int NP2 = (N + 1) / 2;        // DoF pairs
    static constexpr int VOFF = 2 * NP2;           // offset of the velocity half inside a shared-memory row
    F2 c_start, c_gp, c_goal, c_is;                // per-lane partial sums over DoFs (summed horizontally at the end)
    F2 a01, a23, a45;                              // sphere-field sums of the link pairs (weights (1,1) (2,1) (2,1))
    float c_coll, c_self;                          // scalar accumulators (map lookups, self field, generic chains)
    float map_pending;                             // occupancy value gathered at the previous step, not yet accumulated
    unsigned map_pending_u8;                       // same for the byte map: the RAW byte (converted when consumed)
    F2 xpp[NP2], xpv[NP2];                         // previous state

    __device__ __forceinline__ void begin() {
        c_start = c_gp = c_goal = c_is = a01 = a23 = a45 = f2(0.f, 0.f);
        c_coll = c_self = map_pending = 0.f;
        map_pending_u8 = 0u;
    }

    // Panda structure (see fk_panda_origins): sin/cos of the three joint PAIRS packed, scalar chain, link pairs packed.
    // OC > 0: the number of obstacle spheres as a compile-time constant (the loop over them unrolls completely: the run-time loop
    // spends ~25 of the link warps' 280 instructions per step on its 8-way unroll with remainder chain); OC = 0: run-time count.
    template <int OC = 0>
    __device__ __forceinline__ void link_fields(const CostParams<float>& P, const CostSmem<float>& sm, const F2 (&xp)[NP2]) {
        static_assert(CHAIN == 0 || N == 7, "Panda structure has 7 joints");
        if constexpr (CHAIN >= 1) {
            F2 S01, C01, S23, C23, S45, C45;
            link_sincos(xp[0], &S01, &C01);
            link_sincos(xp[1], &S23, &C23);
            link_sincos(xp[2], &S45, &C45);
            const float s0 = lane0(S01), c0 = lane0(C01), s1 = lane1(S01), c1 = lane1(C01);
            // joints 1 and 2 by hand: a = (c1 c0, c1 s0, -s1), b = (-s1 c0, -s1 s0, -c1), c = (-s0, c0, 0), p = (0,0,d1)
            const float d1 = P.p[0][2], t2y = P.p[2][1];
            const float s1c0 = s1 * c0, s1s0 = s1 * s0;
            float X[PANDA_EVAL_LINKS], Y[PANDA_EVAL_LINKS], Z[PANDA_EVAL_LINKS];
            // origins come out in the shifted RBF frame (stage_cta_constants): p - o, folded into the first link offset
            float ox, oy, oz, o_unused;
            load4(sm.sph + SPH_ORIGIN, ox, oy, oz, o_unused);
            float px = fmaf(-t2y, s1c0, -ox), py = fmaf(-t2y, s1s0, -oy), pz = fmaf(-t2y, c1, d1 - oz);
            X[0] = px; Y[0] = py; Z[0] = pz;                                   // link3
            Cols<float> R;
            R.ax = c1 * c0; R.ay = c1 * s0; R.az = -s1;
            R.bx = -s0; R.by = c0; R.bz = 0.f;
            R.cx = s1c0; R.cy = s1s0; R.cz = c1;
            R.rot_z_sc(lane0(S23), lane0(C23));
            px = fmaf(P.p[3][0], R.ax, px); py = fmaf(P.p[3][0], R.ay, py); pz = fmaf(P.p[3][0], R.az, pz);
            X[1] = px; Y[1] = py; Z[1] = pz;                                   // link4
            R.rot_xp90();
            R.rot_z_sc(lane1(S23), lane1(C23));
            px = fmaf(P.p[4][0], R.ax, fmaf(P.p[4][1], R.bx, px));
            py = fmaf(P.p[4][0], R.ay, fmaf(P.p[4][1], R.by, py));
            pz = fmaf(P.p[4][0], R.az, fmaf(P.p[4][1], R.bz, pz));
            X[2] = px; Y[2] = py; Z[2] = pz;                                   // link5 (= link6)
            R.rot_xm90();
            R.rot_z_sc(lane0(S45), lane0(C45));
            R.rot_xp90();
            R.rot_z_sc(lane1(S45), lane1(C45));
            px = fmaf(P.p[6][0], R.ax, px); py = fmaf(P.p[6][0], R.ay, py); pz = fmaf(P.p[6][0], R.az, pz);
            X[3] = px; Y[3] = py; Z[3] = pz;                                   // link7
            px = fmaf(-P.p[7][2], R.bx, px); py = fmaf(-P.p[7][2], R.by, py); pz = fmaf(-P.p[7][2], R.bz, pz);
            X[4] = px; Y[4] = py; Z[4] = pz;                                   // link8 (= hand)
            px = fmaf(-P.p[9][2], R.bx, px); py = fmaf(-P.p[9][2], R.by, py); pz = fmaf(-P.p[9][2], R.bz, pz);
            X[5] = px; Y[5] = py; Z[5] = pz;                                   // ee_link
            // link pairs: (link3, link4) w (1,1); (link5, link7) w (2,1); (link8, ee) w (2,1)
            const F2 X01 = f2(X[0], X[1]), Y01 = f2(Y[0], Y[1]), Z01 = f2(Z[0], Z[1]);
            const F2 X23 = f2(X[2], X[3]), Y23 = f2(Y[2], Y[3]), Z23 = f2(Z[2], Z[3]);
            const F2 X45 = f2(X[4], X[5]), Y45 = f2(Y[4], Y[5]), Z45 = f2(Z[4], Z[5]);
            const F2 P01 = vfma(X01, X01, vfma(Y01, Y01, Z01 * Z01));
            const F2 P23 = vfma(X23, X23, vfma(Y23, Y23, Z23 * Z23));
            const F2 P45 = vfma(X45, X45, vfma(Y45, Y45, Z45 * Z45));
            if (OC > 0 || P.has_spheres) {
                const int O = OC > 0 ? OC : P.n_spheres;
#pragma unroll
                for (int o = 0; o < O; ++o) {
                    const float* s = sm.sph + SPH_STRIDE * o;
                    const float k = s[3];
                    float ax, ay, az, b;
                    load4(s + 4, ax, ay, az, b);
                    a01 += vexp2_fast(vfma(X01, ax, vfma(Y01, ay, vfma(Z01, az, vfma(P01, k, b)))));
                    a23 += vexp2_fast(vfma(X23, ax, vfma(Y23, ay, vfma(Z23, az, vfma(P23, k, b)))));
                    a45 += vexp2_fast(vfma(X45, ax, vfma(Y45, ay, vfma(Z45, az, vfma(P45, k, b)))));
                }
            }
            if (CHAIN == 2 && P.has_self) {
                const float ks = P.self_k, z0 = P.p[0][2];
                float PP[PANDA_EVAL_LINKS] = {lane0(P01), lane1(P01), lane0(P23), lane1(P23), lane0(P45), lane1(P45)};
                float w1 = 0.f, w2 = 0.f, w4 = 0.f;     // sums of E over unordered pairs with weight product 1, 2, 4
#pragma unroll
                for (int l = 0; l < PANDA_EVAL_LINKS; ++l) {
                    const bool l2 = (l == 2 || l == 4);
                    const float e12 = vexp2_fast(ks * fmaf(-2.f * z0, Z[l], PP[l] + z0 * z0));
                    if (l2) w4 += e12; else w2 += e12;
                    if (P.include_base) {
                        const float eb = vexp2_fast(ks * PP[l]);
                        if (l2) w2 += eb; else w1 += eb;
                    }
#pragma unroll
                    for (int m = l + 1; m < PANDA_EVAL_LINKS; ++m) {
                        const float dx = X[l] - X[m], dy = Y[l] - Y[m], dz = Z[l] - Z[m];
                        const float e = vexp2_fast(ks * fmaf(dx, dx, fmaf(dy, dy, dz * dz)));
                        const int wp = (l2 ? 2 : 1) * ((m == 2 || m == 4) ? 2 : 1);
                        if (wp == 4) w4 += e; else if (wp == 2) w2 += e; else w1 += e;
                    }
                }
                c_self += 2.f * (w1 + (2.f * w2 + 4.f * w4));
            }
        }
    }

    // Issues the gather of this step and accumulates the one of the PREVIOUS step: nothing in this step depends on the
    // load (not even the byte -> float conversion), so its L1/L2 latency hides behind the next step's RNG and recurrence
    // (ncu: the gather's consumer carried 23 % of the planar kernel's stall samples).  Occupancy sums are small integers,
    // exact in any order: bit-identical to the in-order sum.
    // MODE 0: byte or float map decided at run time; 1: byte map; 2: float map (the state-only fused kernel picks the mode once
    // per sweep, so the per-step pointer test and the predicated twin of the gather disappear from its hot loop)
    template <int MODE = 0>
    __device__ __forceinline__ void map_gather_deferred(const CostParams<float>& P, const CostSmem<float>& sm, float x, float y) {
        const float xo = sg_mul_add_2r(x, P.map_inv_cell, P.map_origin_x);
        const float yo = sg_mul_add_2r(y, P.map_inv_cell, P.map_origin_y);
        int ix = (int)floorf(xo), iy = (int)floorf(yo);
        ix = min(max(ix, 0), P.map_h - 1);
        iy = min(max(iy, 0), P.map_w - 1);
        const int idx = iy * P.map_w + ix;
        if (MODE == 1 || (MODE == 0 && sm.map_u8)) {
            c_coll += (float)map_pending_u8;
            map_pending_u8 = __ldg(sm.map_u8 + idx);
        } else {
            c_coll += map_pending;
            map_pending = __ldg(sm.map + idx);
        }
    }

    // feed state x_t as DoF pairs: xp[k] = (pos_2k, pos_2k+1), xv[k] = (vel_2k, vel_2k+1)
    // srow / grow / brow: start, goal and b_t rows in the pair layout [pos pairs][vel pairs] (16-byte aligned)
    // yp / yv: the deviations x - mu (IS term = mu^T b + y^T b, see TrajCost::step)
    __device__ __forceinline__ void step(const CostParams<float>& P, const CostSmem<float>& sm, int t, int T,
                                         const F2 (&xp)[NP2], const F2 (&xv)[NP2], const F2 (&yp)[NP2], const F2 (&yv)[NP2],
                                         const float* brow) {
        auto pair_at = [](const float* row, int k) { return f2(row[2 * k], row[2 * k + 1]); };   // folds into LDS.64/128
        if (t == 0) {
#pragma unroll
            for (int k = 0; k < NP2; ++k) {
                const F2 ep = pair_at(sm.start, k) - xp[k], ev = pair_at(sm.start + VOFF, k) - xv[k];
                c_start = vfma(ep, ep, vfma(ev, ev, c_start));
            }
        } else {
#pragma unroll
            for (int k = 0; k < NP2; ++k) {
                const F2 ep = vfma(-P.dt, xpv[k], xp[k] - xpp[k]);
                const F2 ev = xv[k] - xpv[k];
                c_gp = vfma(ep, vfma(P.q12x2, ev, P.q11 * ep), c_gp);
                c_gp = vfma(P.q22 * ev, ev, c_gp);
            }
            if (P.has_map) map_gather_deferred(P, sm, lane0(xp[0]), lane1(xp[0]));
            if (CHAIN >= 1 && (P.has_spheres || P.has_self)) link_fields(P, sm, xp);
        }
        if (t == T - 1 && P.has_goal) {
#pragma unroll
            for (int k = 0; k < NP2; ++k) {
                const F2 ep = pair_at(sm.goal, k) - xp[k], ev = pair_at(sm.goal + VOFF, k) - xv[k];
                c_goal = vfma(ep, ep, vfma(ev, ev, c_goal));
            }
        }
        if (brow) {
#pragma unroll
            for (int k = 0; k < NP2; ++k) c_is = vfma(yp[k], pair_at(brow, k), vfma(yv[k], pair_at(brow + VOFF, k), c_is));
        }
#pragma unroll
        for (int k = 0; k < NP2; ++k) { xpp[k] = xp[k]; xpv[k] = xv[k]; }
    }

    __device__ __forceinline__ float total(const CostParams<float>& P, const CostSmem<float>& sm, int T, float* terms6) {
        const float st = hsum(c_start) * P.inv_sig_start2;
        const float gp = hsum(c_gp);
        const float go = hsum(c_goal) * P.inv_sig_goal2;
        float coll = (c_coll + map_pending) + (float)map_pending_u8, self = c_self;
        if (CHAIN >= 1) {
            coll += (hsum(a01) + (2.f * lane0(a23) + lane1(a23))) + (2.f * lane0(a45) + lane1(a45));
            coll += (float)(T - 1) * sm.coll_const;
            self += (float)(T - 1) * sm.self_const;
        }
        coll *= (P.has_map ? P.map_w_coll : P.sphere_w_coll);
        self *= P.self_w_coll;
        const float is = (hsum(c_is) + sm.mub) * P.temperature;
        float ee = 0.f;
        if (P.has_ee) {     // EE SE(3) goal on the last state (xpp holds the positions of x_{T-1})
            float q[2 * NP2];
#pragma unroll
            for (int k = 0; k < NP2; ++k) { q[2 * k] = lane0(xpp[k]); q[2 * k + 1] = lane1(xpp[k]); }
            ee = ee_se3_cost<float, N>(P, q) * P.ee_w;
        }
        if (terms6) { terms6[0] = st; terms6[1] = gp; terms6[2] = go; terms6[3] = coll; terms6[4] = is; terms6[5] = self; }
        return (((((st + gp) + go) + self) + coll) + ee) + is;
    }
};

}  // namespace sgpmp
