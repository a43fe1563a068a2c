// Fused StochGPMP iteration for the Panda structure, ROLE-SPLIT across warps (fp32, 7 DoF, RBF link fields).
// Same contract as iterate_kernel (sgpmp_iterate.cu): sample -> cost -> softmax -> weighted update, n_iters times in
// one launch; replaces planner.py:239-275 per iteration.  What changes is who does what inside pass 1:
//
//   * STATE warps (role A) own the sequential part of a trajectory sample: Philox/Box-Muller normals, the banded
//     recurrence y_t = G_t eps_t - H_t y_{t-1}, the GP / start / goal factors and the importance-sampling dot.
//     The GP error is formed from the DEVIATIONS:  e_t = (y_t - Phi y_{t-1}) + (mu_t - Phi mu_{t-1}), the second
//     term staged per particle in shared memory (computed in fp64 once per iteration) — no previous-state
//     registers, no velocity states, and an order of magnitude less fp32 cancellation than differencing x_t.
//   * LINK warps (role B) own the part that is a pure function of q_t: sin/cos, the structured Panda chain
//     (fk_panda_origins), the sphere RBF field and the self-collision field (TrajCostPairs::link_fields).
//   * The only thing that crosses is q_t[0..5] — 24 bytes per (sample, step) — through a shared-memory ring
//     (NSTG stages of TS steps per warp pair), handed over with mbarriers (full / empty, 32 arrivals each).
//     State warp w feeds link warp w: same 32 samples, lane to lane, so no __syncthreads exists inside pass 1.
//
// Why: the single-role kernel keeps both halves' live state in one thread (80 registers at 3 CTAs/SM, 3 % of its
// instructions are spills, RNG and FK compete for the same registers and instruction cache).  Split, each role
// fits 64 registers without spills, the SM holds 32 warps instead of 24, and the scheduler always has an ALU/XU
// stream (Philox, Box-Muller) next to an FMA/XU stream (chain, RBF) to pick from.  See DESIGN.md §4.2.
#include <type_traits>

#include "sgpmp_common.cuh"
#include "sgpmp_cost.cuh"
#include "sgpmp_cost_pairs.cuh"
#include "sgpmp_iterate.cuh"
#include "sgpmp_rng.cuh"

namespace sgpmp {

constexpr int SPLIT_TS = 5;     // time steps per ring stage (C4: 1 / 2 / 3 / 4 / 5 steps 13.77 / 13.62 / 13.32 / 13.21 / 13.11 ms; 6 no longer fits four CTAs per SM)
constexpr int SPLIT_NSTG = 2;   // ring stages per warp pair

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Wait until the phase of the given parity has completed (a fresh barrier has "completed" parity 1).  A warp that has to
// wait is SUSPENDED: a spinning warp would spend the issue slots the other role needs (first version: 7 % of all executed
// instructions were this loop).  The hardware suspends the warp inside try_wait for up to the hinted time, so no instructions
// run between polls.  Measured at C4 (profiles/r2/wait_variants.txt): hint 1000 / 20000 ns 13.15 ms, try_wait + nanosleep
// 64 / 256 / 1000 / 4000 ns 13.21-13.22 ms — the wait loop is not what bounds the kernel (a waiting warp only uses issue slots
// nobody else had a use for).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    constexpr uint32_t HINT_NS = 1000;
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(bar)), "r"(parity), "r"(HINT_NS)
        : "memory");
}

__device__ __forceinline__ F2 ld_f2(const float* p) { const float2 v = *reinterpret_cast<const float2*>(p); return f2(v.x, v.y); }
__device__ __forceinline__ F2 ld_f2(const float2* p) { const float2 v = *p; return f2(v.x, v.y); }
__device__ __forceinline__ void st_f2(float2* p, F2 v) { *p = make_float2(lane0(v), lane1(v)); }
__device__ __forceinline__ void ld_2f2(const float* p, F2& a, F2& b) {     // one LDS.128 -> two packed pairs
    const float4 v = *reinterpret_cast<const float4*>(p);
    a = f2(v.x, v.y); b = f2(v.z, v.w);
}

// Per-time-step record of a particle in shared memory, laid out in the order the state warps consume it:
//   [0..7]             g11 g21 g22 -h11 | -h12 -h21 -h22 0          (H stored negated: y_t = G eps_t + (-H) y_{t-1})
//   [8 + 12k .. +11]   DoF pair k:  gmu (p0 p1 v0 v1) | b (p0 p1 v0 v1) | mu (p0 p1 v0 v1)
// gmu = mu_t - Phi mu_{t-1} (GP residual of the mean), b = Sigma^-1 mu.  One pointer walks it, every access is an
// LDS.128/LDS.64 at an immediate offset.  The ghost DoF (odd count) holds zeros.
constexpr int REC_G = 0, REC_B = 4, REC_M = 8;
__host__ __device__ constexpr int rec_floats(int n_dof) { return 8 + 12 * ((n_dof + 1) / 2); }
__device__ __forceinline__ int rec_col(int i, int a, int what) { return 8 + 12 * (i >> 1) + what + 2 * a + (i & 1); }   // a: 0 pos, 1 vel

// NA state warps + NB link warps per CTA: 32 NA samples per sweep.  NB = NA: state warp w feeds link warp w.  NB = 0: no link
// fields (CHAIN = 0; the planar occupancy-map cost is gathered by the state warps themselves) — then there is no ring and no
// mbarrier, just the state role with its record layout.
template <int NA, int NB> struct SplitCfg {
    static_assert(NB == 0 || NB == NA, "one link warp per state warp");
    static constexpr int BS = 32 * (NA + NB), SW = 32 * NA;
    // CTAs per SM: with link warps as many as 1024 threads (64 registers each) allow; state-only CTAs fit 48 registers
    static constexpr int MINB = NB ? 1024 / BS : (1280 / BS > 24 ? 24 : 1280 / BS);
    // shared-memory bytes of the region that pass 1 uses for the ring + link sums and the block phases for acc / nzl / nzo
    __host__ __device__ static constexpr size_t pass1_bytes() {
        return NB ? (size_t)NA * SPLIT_NSTG * SPLIT_TS * 96 * sizeof(float2) + (size_t)32 * NA * 8 * sizeof(float) : 0;
    }
};

template <int N, int CHAIN, int NA, int NB>
__global__ void __launch_bounds__(SplitCfg<NA, NB>::BS, SplitCfg<NA, NB>::MINB)
iterate_split_kernel(const __grid_constant__ CostParams<float> P, const __grid_constant__ IterArgs<float> A) {
    using Cfg = SplitCfg<NA, NB>;
    constexpr int d = 2 * N, NP2 = (N + 1) / 2, REC = rec_floats(N), BS = Cfg::BS, SW = Cfg::SW;
    static_assert((CHAIN == 0) == (NB == 0), "link warps exist exactly when the chain has link fields");
    static_assert(CHAIN == 0 || N == 7, "Panda structure has 7 joints");
    static_assert(NP2 <= 4, "start / goal staging holds up to 8 DoF");
    constexpr int TS = NB ? SPLIT_TS : 16;      // state-only form: a 'stage' is just the span of the two-level GP sum
    constexpr int NSTG = SPLIT_NSTG;
    constexpr int SLOT = 3 * 32;                                      // float2 per (state warp, step): q pairs 0..2 x 32 lanes
    const int T = A.T, S = A.S, G = A.G, K = A.K;
    const int M = T * d, Mpad = (M + 3) & ~3, Spad = (S + 3) & ~3, NCH = (S + 31) >> 5;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* sph = reinterpret_cast<float*>(smem_raw);           // [MAX_SPHERES][8] + coll_const, self_const
    float* rec = sph + SPH_SMEM;                               // [T][REC]
    float* wsm = rec + (size_t)T * REC;                        // [S] costs -> weights
    float* red = wsm + Spad;                                   // [32]
    float* start = red + 32;                                   // [16] pair-interleaved like the mu block of a record
    float* goal = start + 16;                                  // [16]
    double* red64 = reinterpret_cast<double*>(goal + 16);      // [32]
    uint64_t* bars = reinterpret_cast<uint64_t*>(red64 + 32);  // [NA][2 NSTG + 1]  (NB > 0)
    unsigned char* uni = reinterpret_cast<unsigned char*>(bars + (NB ? ((NA * (2 * NSTG + 1) + 1) & ~1) : 0));
    // -- the union region: pass 1 ...
    float2* ring = reinterpret_cast<float2*>(uni);             // [NA][NSTG][TS][3][32]
    float* bacc = reinterpret_cast<float*>(ring + (size_t)NA * NSTG * TS * SLOT);   // [32 NA][8] link-field sums of a sweep
    // -- ... and the block phases
    float* acc = reinterpret_cast<float*>(uni);                // [T][d] sum_s w_s eps_s, then grad
    int* nzl = reinterpret_cast<int*>(acc + Mpad);             // [S] samples with non-zero weight, in order
    int* nzo = nzl + Spad;                                     // [NCH + 1] their per-32-chunk offsets
    float* stg_tmp = acc;                                      // [32] staging scratch at start-up

    const int NP = G * K;
    const int bp = blockIdx.x, b = bp / NP, p = bp - b * NP;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int role = warp < NA ? 0 : 1;                         // 0: state warps, 1: link warps
    const int wa = warp, wb = warp - NA;
    const uint32_t pgid = A.particle_gid0 + (uint32_t)bp;
    auto bar_full = [&](int w, uint32_t stg) { return bars + w * (2 * NSTG + 1) + stg; };
    auto bar_empty = [&](int w, uint32_t stg) { return bars + w * (2 * NSTG + 1) + NSTG + stg; };
    auto bar_res = [&](int w) { return bars + w * (2 * NSTG + 1) + 2 * NSTG; };
    auto pidx = [](int j) { return (j < N ? rec_col(j, 0, 0) : rec_col(j - N, 1, 0)) - 8; };   // state index -> column of a pair block

    if (NB > 0 && tid < NA * (2 * NSTG + 1)) mbar_init(bars + tid, 32);
    for (int k = tid; k < T * REC; k += BS) rec[k] = 0.f;
    __syncthreads();
    for (int k = tid; k < T * 8; k += BS) {
        const int t = k >> 3, c = k & 7;
        const double* row = A.tab + (size_t)t * SGPMP_TABLE_STRIDE;
        rec[t * REC + c] = c < 3 ? (float)row[c] : (c < 7 ? -(float)row[c] : 0.f);
    }
    for (int k = tid; k < M; k += BS) {
        const int t = k / d, j = k - t * d;
        rec[t * REC + REC_M + 8 + pidx(j)] = A.means[(size_t)bp * M + k];
    }
    stage_cta_constants<float, N, CHAIN, 2 * NP2>(P, b, p / K, G, stg_tmp, stg_tmp + 16, sph);
    if (tid < 32) {      // re-lay start / goal from [pos pairs | vel pairs] to the pair-interleaved order (stage_cta_constants ended with a barrier)
        const int i = tid & 7, a = (tid >> 3) & 1, which = tid >> 4;
        if (i < 2 * NP2) (which ? goal : start)[4 * (i >> 1) + 2 * a + (i & 1)] = stg_tmp[16 * which + 2 * NP2 * a + i];
    }
    CostSmem<float> sm;
    sm.start = start; sm.goal = goal; sm.bvec = nullptr; sm.sph = sph;
    sm.coll_const = sph[SPH_STRIDE * SGPMP_MAX_SPHERES];
    sm.self_const = sph[SPH_STRIDE * SGPMP_MAX_SPHERES + 1];
    sm.map = P.has_map ? P.occ_map + (size_t)(P.map_of_problem ? P.map_of_problem[b] : 0) * P.map_h * P.map_w : nullptr;
    sm.map_u8 = (P.has_map && P.occ_map_u8) ? P.occ_map_u8 + (size_t)(P.map_of_problem ? P.map_of_problem[b] : 0) * P.map_h * P.map_w : nullptr;
    __syncthreads();

    const int ns = S;
    const int n_sweeps = (ns + SW - 1) / SW;
    uint32_t sc = 0;      // ring stages used so far (identical in both roles)
    uint32_t rc = 0;      // sweeps finished so far

    for (int it = 0; it < A.n_iters; ++it) {
        const bool last = (it == A.n_iters - 1);
        const RngKey& key = A.key;
        const uint32_t dro = (uint32_t)it;      // draw index of this iteration = key.draw + it
        const float* eps = A.eps_in ? A.eps_in + ((size_t)it * gridDim.x + bp) * (size_t)M * S : nullptr;

        // ---- b = Sigma^-1 mu (arithmetic of precision_times_row, sgpmp_cost.cuh) and the GP residual of the mean, fp64 ----
        double mub_part = 0.0;
        for (int k = tid; k < T * N; k += BS) {
            const int t = k / N, i = k - t * N;
            float* blk = rec + t * REC;
            const int cp = rec_col(i, 0, 0), cv = rec_col(i, 1, 0);
            const double* r = A.tab + (size_t)t * SGPMP_TABLE_STRIDE + SGPMP_TAB_D11;     // (d11 d12 d22 o11 o12 o21 o22) of step t
            const double mp = blk[cp + REC_M], mv = blk[cv + REC_M];
            double bp_ = r[0] * mp + r[1] * mv;
            double bv_ = r[1] * mp + r[2] * mv;
            if (t > 0) {
                const double* q = r - SGPMP_TABLE_STRIDE;
                const double ap = blk[cp + REC_M - REC], av = blk[cv + REC_M - REC];
                bp_ += q[3] * ap + q[4] * av;
                bv_ += q[5] * ap + q[6] * av;
                blk[cp + REC_G] = (float)((mp - ap) - (double)P.dt * av);
                blk[cv + REC_G] = (float)(mv - av);
            }
            if (t < T - 1) {
                const double ap = blk[cp + REC_M + REC], av = blk[cv + REC_M + REC];
                bp_ += r[3] * ap + r[5] * av;   // O_t^T
                bv_ += r[4] * ap + r[6] * av;
            }
            blk[cp + REC_B] = (float)bp_;
            blk[cv + REC_B] = (float)bv_;
            mub_part += mp * bp_ + mv * bv_;
        }
        const float mub = (float)block_sum_f64(mub_part, red64);
        if (last && A.means_pre)
            for (int k = tid; k < M; k += BS) A.means_pre[(size_t)bp * M + k] = rec[(k / d) * REC + REC_M + 8 + pidx(k % d)];
        __syncthreads();

        // ---- pass 1 -------------------------------------------------------------------------------------
        const bool emit = last && A.samples != nullptr;
        for (int sw = 0; sw < n_sweeps; ++sw) {
            if (role == 0) {
              // MM: occupancy-map mode of this sweep — -1 none, 1 byte map, 2 float map (state-only form; a compile-time constant of
              // the time loop instead of a per-step test)
              auto state_sweep = [&](auto mm_) {
                constexpr int MM = decltype(mm_)::value;
                const int sl = sw * SW + wa * 32 + lane;
                const bool valid = sl < ns;
                const int s0 = valid ? sl : ns - 1;              // idle lanes shadow the last sample, results dropped
                // ================= state warps =================
                const uint32_t sgid = A.sample_gid0 + (uint32_t)s0;
                F2 yp[NP2], yv[NP2];
#pragma unroll
                for (int k = 0; k < NP2; ++k) yp[k] = yv[k] = f2(0.f, 0.f);
                F2 cgp = f2(0.f, 0.f), cis = f2(0.f, 0.f), cst = f2(0.f, 0.f), cgo = f2(0.f, 0.f);
                TrajCostPairs<N, 0> tcm;          // occupancy-map gather of the state warps (planar: obst_map.py:164-182)
                tcm.begin();
                auto draw = [&](int t, F2 (&ep)[NP2], F2 (&ev)[NP2]) {
                    if (eps) {
                        const float* r0 = eps + ((size_t)t * d) * S + s0;
#pragma unroll
                        for (int k = 0; k < NP2; ++k) {
                            const int i0 = 2 * k, i1 = 2 * k + 1;
                            ep[k] = f2(r0[(size_t)i0 * S], i1 < N ? r0[(size_t)i1 * S] : 0.f);
                            ev[k] = f2(r0[(size_t)(N + i0) * S], i1 < N ? r0[(size_t)(N + i1) * S] : 0.f);
                        }
                    } else {
#pragma unroll
                        for (int k = 0; k < NP2; ++k) {
                            if (2 * k + 1 < N) normal_pair_f2<true>(key, (uint32_t)t, (uint32_t)k, sgid, pgid, ep[k], ev[k], dro);
                            else normal_pair_f2<false>(key, (uint32_t)t, (uint32_t)k, sgid, pgid, ep[k], ev[k], dro);
                        }
                    }
                };
                auto emit_row = [&](int t) {      // last iteration only: x_t = mu_t + y_t to global memory
                    const float* blk = rec + t * REC + 8;
                    float* row = A.samples + ((size_t)bp * M + (size_t)t * d) * S + s0;
#pragma unroll
                    for (int k = 0; k < NP2; ++k) {
                        F2 mp, mv;
                        ld_2f2(blk + 12 * k + REC_M, mp, mv);
                        const F2 xp = mp + yp[k], xv = mv + yv[k];
                        row[(size_t)(2 * k) * S] = lane0(xp);
                        row[(size_t)(N + 2 * k) * S] = lane0(xv);
                        if (2 * k + 1 < N) { row[(size_t)(2 * k + 1) * S] = lane1(xp); row[(size_t)(N + 2 * k + 1) * S] = lane1(xv); }
                    }
                };
                {   // t = 0: start factor (cost_functions.py:131-134); no GP error, no collision term (traj_range [1, T))
                    F2 ep[NP2], ev[NP2];
                    draw(0, ep, ev);
                    float r[8];
                    load4(rec, r[0], r[1], r[2], r[3]);
                    load4(rec + 4, r[4], r[5], r[6], r[7]);
#pragma unroll
                    for (int k = 0; k < NP2; ++k) {
                        F2 bp_, bv_, mp, mv, sp, sv;
                        ld_2f2(rec + 8 + 12 * k + REC_B, bp_, bv_);
                        ld_2f2(rec + 8 + 12 * k + REC_M, mp, mv);
                        ld_2f2(start + 4 * k, sp, sv);
                        yp[k] = r[0] * ep[k];
                        yv[k] = vfma(r[1], ep[k], r[2] * ev[k]);
                        const F2 dp = sp - (mp + yp[k]);
                        const F2 dv = sv - (mv + yv[k]);
                        cst = vfma(dp, dp, vfma(dv, dv, cst));
                        cis = vfma(yp[k], bp_, vfma(yv[k], bv_, cis));
                    }
                    if (emit && valid) emit_row(0);
                }
                for (int t0 = 1; t0 < T; t0 += TS) {
                    const uint32_t stg = sc % NSTG, use = sc / NSTG;
                    if constexpr (NB > 0) mbar_wait(bar_empty(wa, stg), (use & 1u) ^ 1u);
                    const int tend = min(t0 + TS, T);
                    float2* slot = NB > 0 ? ring + ((size_t)(wa * NSTG + stg) * TS) * SLOT + lane : nullptr;
                    const float* blk = rec + t0 * REC;
                    F2 cgs = f2(0.f, 0.f);          // GP sum of this stage (two-level accumulation)
#pragma unroll 1
                    for (int t = t0; t < tend; ++t, slot += SLOT, blk += REC) {
                        F2 ep[NP2], ev[NP2];
                        draw(t, ep, ev);
                        float r[8];
                        load4(blk, r[0], r[1], r[2], r[3]);
                        load4(blk + 4, r[4], r[5], r[6], r[7]);
#pragma unroll
                        for (int k = 0; k < NP2; ++k) {
                            F2 gp_, gv_, bp_, bv_;
                            ld_2f2(blk + 8 + 12 * k + REC_G, gp_, gv_);
                            ld_2f2(blk + 8 + 12 * k + REC_B, bp_, bv_);
                            // everything that needs y_{t-1} first, so that y_t can be formed IN PLACE (no loop-carried copies):
                            //   t_ = -H11 yp - H12 yv, u_ = -H21 yp - H22 yv, w_ = yp + dt yv (= Phi y_{t-1}, position row), z_ = gmu_v - yv
                            const F2 t_ = vfma(r[3], yp[k], r[4] * yv[k]);
                            const F2 u_ = vfma(r[5], yp[k], r[6] * yv[k]);
                            const F2 w_ = vfma(P.dt, yv[k], yp[k]);
                            const F2 z_ = gv_ - yv[k];
                            yp[k] = vfma(r[0], ep[k], t_);
                            yv[k] = vfma(r[1], ep[k], vfma(r[2], ev[k], u_));
                            // GP factor on the deviations (gp_factor.py:54-58): e = (y_t - Phi y_{t-1}) + (mu_t - Phi mu_{t-1})
                            const F2 e_p = (yp[k] - w_) + gp_;
                            const F2 e_v = yv[k] + z_;
                            cgs = vfma(e_p, vfma(P.q12x2, e_v, P.q11 * e_p), cgs);
                            cgs = vfma(P.q22 * e_v, e_v, cgs);
                            cis = vfma(yp[k], bp_, vfma(yv[k], bv_, cis));
                            if (NB > 0 && k < 3) st_f2(slot + 32 * k, ld_f2(blk + 8 + 12 * k + REC_M) + yp[k]);   // q_t[2k], q_t[2k+1] for the link warp
                        }
                        if constexpr (NB == 0 && MM > 0) {
                            const F2 x01 = ld_f2(blk + 8 + REC_M) + yp[0];
                            tcm.template map_gather_deferred<MM>(P, sm, lane0(x01), lane1(x01));
                        }
                        if (emit && valid) emit_row(t);
                    }
                    cgp += cgs;
                    if constexpr (NB > 0) mbar_arrive(bar_full(wa, stg));
                    ++sc;
                }
                // goal prior on x_{T-1} (cost_functions.py:376-388) and the EE SE(3) goal (cost_functions.py:308-321)
                const float* mlast = rec + (T - 1) * REC + 8 + REC_M;
                if (P.has_goal) {
#pragma unroll
                    for (int k = 0; k < NP2; ++k) {
                        F2 mp, mv, gp_, gv_;
                        ld_2f2(mlast + 12 * k, mp, mv);
                        ld_2f2(goal + 4 * k, gp_, gv_);
                        const F2 dp = gp_ - (mp + yp[k]);
                        const F2 dv = gv_ - (mv + yv[k]);
                        cgo = vfma(dp, dp, vfma(dv, dv, cgo));
                    }
                }
                float ee = 0.f;
                if (N == 7 && P.has_ee) {
                    float q[2 * NP2];
#pragma unroll
                    for (int k = 0; k < NP2; ++k) {
                        const F2 x = ld_f2(mlast + 12 * k) + yp[k];
                        q[2 * k] = lane0(x); q[2 * k + 1] = lane1(x);
                    }
                    ee = ee_se3_cost<float, N>(P, q) * P.ee_w;
                }
                const float st = hsum(cst) * P.inv_sig_start2;
                const float gp = hsum(cgp);
                const float go = hsum(cgo) * P.inv_sig_goal2;
                const float is = (hsum(cis) + mub) * P.temperature;
                float coll, self = 0.f;
                if constexpr (NB > 0) {
                    mbar_wait(bar_res(wa), rc & 1u);
                    const float4* ba = reinterpret_cast<const float4*>(bacc + (size_t)(wa * 32 + lane) * 8);
                    const float4 v0 = ba[0], v1 = ba[1];       // link pairs (l3, l4) (l5, l7) | (l8, ee) self -
                    coll = ((v0.x + v0.y) + (2.f * v0.z + v0.w)) + (2.f * v1.x + v1.y);
                    coll += (float)(T - 1) * sm.coll_const;
                    coll *= P.sphere_w_coll;
                    self = (v1.z + (float)(T - 1) * sm.self_const) * P.self_w_coll;
                } else {
                    coll = ((tcm.c_coll + tcm.map_pending) + (float)tcm.map_pending_u8) * P.map_w_coll;     // 0 without a map
                }
                // summation order of the shipped cost lists: CostGP (start + gp), CostGoalPrior, self-collision, obstacle
                // collision, EE goal (examples/panda_environment.py:90), then += IS (planner.py:236)
                const float c = (((((st + gp) + go) + self) + coll) + ee) + is;
                if (valid) {
                    wsm[sl] = c;
                    if (last && A.costs) A.costs[(size_t)bp * S + sl] = c;
                }
              };
              if constexpr (NB == 0) {
                  if (!P.has_map) state_sweep(std::integral_constant<int, -1>{});
                  else if (sm.map_u8) state_sweep(std::integral_constant<int, 1>{});
                  else state_sweep(std::integral_constant<int, 2>{});
              } else {
                  state_sweep(std::integral_constant<int, -1>{});
              }
            } else if constexpr (NB > 0) {
                // ================= link warps =================
                // Link warp wb serves state warp wb.  The field sums of the whole sweep stay in registers and reach shared memory
                // once, at the end (folding them into shared memory per stage cost ~16 instructions per stage on the warps that
                // are the critical path).  The sweep is instantiated for the common sphere counts as compile-time constants
                // (oc = 0: run-time loop).
                auto link_sweep = [&](auto oc) {
                    constexpr int OC = decltype(oc)::value;
                    TrajCostPairs<N, CHAIN> tc;
                    tc.begin();
                    for (int t0 = 1; t0 < T; t0 += TS) {
                        const uint32_t stg = sc % NSTG, use = sc / NSTG;
                        const int tend = min(t0 + TS, T);
                        mbar_wait(bar_full(wb, stg), use & 1u);
                        const float2* slot = ring + ((size_t)(wb * NSTG + stg) * TS) * SLOT + lane;
#pragma unroll 1
                        for (int t = t0; t < tend; ++t, slot += SLOT) {
                            F2 xq[NP2];
                            xq[0] = ld_f2(slot); xq[1] = ld_f2(slot + 32); xq[2] = ld_f2(slot + 64);
                            xq[3] = f2(0.f, 0.f);
                            tc.template link_fields<OC>(P, sm, xq);
                        }
                        mbar_arrive(bar_empty(wb, stg));
                        ++sc;
                    }
                    float4* ba = reinterpret_cast<float4*>(bacc + (size_t)(wb * 32 + lane) * 8);
                    ba[0] = make_float4(lane0(tc.a01), lane1(tc.a01), lane0(tc.a23), lane1(tc.a23));
                    ba[1] = make_float4(lane0(tc.a45), lane1(tc.a45), tc.c_self, 0.f);
                    mbar_arrive(bar_res(wb));                            // the sums of the sweep are complete
                };
                const int n_sph = P.has_spheres ? P.n_spheres : -1;
                if (n_sph == 5) link_sweep(std::integral_constant<int, 5>{});          // examples/panda_environment.py:125-133
                else if (n_sph == 4) link_sweep(std::integral_constant<int, 4>{});
                else if (n_sph == 8) link_sweep(std::integral_constant<int, 8>{});
                else link_sweep(std::integral_constant<int, 0>{});
            }
            ++rc;
        }
        __syncthreads();

        // ---- softmax over the S samples of this particle ------------------------------------------------
        float smax, ssum;
        {
            float m = -INFINITY;
            for (int s = tid; s < ns; s += BS) {
                const float z = -wsm[s] / P.temperature;
                wsm[s] = z;
                m = fmaxf(m, z);
            }
            m = warp_max(m);
            if (lane == 0) red[warp] = m;
            __syncthreads();
            m = red[0];
            for (int k = 1; k < BS / 32; ++k) m = fmaxf(m, red[k]);
            __syncthreads();
            float Z = 0;
            for (int s = tid; s < ns; s += BS) {
                const float ex = sg_exp(wsm[s] - m);
                wsm[s] = ex;
                Z += ex;
            }
            Z = warp_sum(Z);
            if (lane == 0) red[warp] = Z;
            __syncthreads();
            Z = 0;
            for (int k = 0; k < BS / 32; ++k) Z += red[k];
            smax = m; ssum = Z;
            // weights, and per 32-sample chunk the number of non-zero ones (the shipped configurations are one-hot)
            for (int c = warp; c < NCH; c += BS / 32) {
                const int s = c * 32 + lane;
                float w = 0.f;
                if (s < ns) {
                    // split-particle mode (stats_out): the weights stay UNNORMALISED, (m, Z) go out with A
                    w = A.stats_out ? wsm[s] : wsm[s] / Z;
                    wsm[s] = w;
                    if (last && A.weights) A.weights[(size_t)bp * S + s] = w;
                }
                const unsigned mask = __ballot_sync(0xffffffffu, w != 0.f);
                if (lane == 0) nzo[c + 1] = __popc(mask);
            }
            __syncthreads();
            if (tid == 0) {
                int run = 0;
                nzo[0] = 0;
                for (int c = 1; c <= NCH; ++c) { run += nzo[c]; nzo[c] = run; }
            }
            __syncthreads();
            for (int c = warp; c < NCH; c += BS / 32) {
                const int s = c * 32 + lane;
                const bool nz = s < ns && wsm[s] != 0.f;
                const unsigned mask = __ballot_sync(0xffffffffu, nz);
                if (nz) nzl[nzo[c] + __popc(mask & ((1u << lane) - 1u))] = s;
            }
            __syncthreads();
        }

        // ---- pass 2: acc = sum_s w_s eps_s over the samples with w_s != 0, in sample order (regenerated from the
        //      counter-based stream with the transposed mapping thread <-> (time step, DoF pair)) ----------------
        if (eps) {
            for (int r = warp; r < M; r += BS / 32) {
                float a = 0;
                for (int s = lane; s < ns; s += 32) a += wsm[s] * eps[(size_t)r * S + s];
                a = warp_sum(a);
                if (lane == 0) acc[r] = a;
            }
        } else {
            const int n_items = T * NP2, nnz = nzo[NCH];
            for (int item = tid; item < n_items; item += BS) {
                const int t_ = item / NP2, k = item - t_ * NP2;
                const bool full = 2 * k + 1 < N;
                float a0 = 0, a1 = 0, a2 = 0, a3 = 0;
                for (int j = 0; j < nnz; ++j) {
                    const int s = nzl[j];
                    const float w = wsm[s];
                    float p0, p1, v0, v1;
                    normal_pair<float>(key, (uint32_t)t_, (uint32_t)k, full, A.sample_gid0 + (uint32_t)s, pgid, p0, p1, v0, v1, dro);
                    a0 += w * p0; a1 += w * p1; a2 += w * v0; a3 += w * v1;
                }
                acc[t_ * d + 2 * k] = a0;
                acc[t_ * d + N + 2 * k] = a2;
                if (full) {
                    acc[t_ * d + 2 * k + 1] = a1;
                    acc[t_ * d + N + 2 * k + 1] = a3;
                }
            }
        }
        __syncthreads();

        if (A.stats_out) {       // split-particle mode: hand (m, Z, A = sum_s exp(z_s - m) eps_s) to the exchange, no update here
            if (tid == 0) { A.stats_out[(size_t)bp * (M + 2)] = smax; A.stats_out[(size_t)bp * (M + 2) + 1] = ssum; }
            for (int k = tid; k < M; k += BS) A.stats_out[(size_t)bp * (M + 2) + 2 + k] = acc[k];
            return;
        }
        // ---- grad = L acc (banded recurrence, one thread per DoF); mu += step * grad --------------------
        if (tid < N) {
            const int i = tid;
            const int cp = rec_col(i, 0, REC_M), cv = rec_col(i, 1, REC_M);
            float gp_ = 0, gv_ = 0;
            for (int t = 0; t < T; ++t) {
                float* r = rec + t * REC;
                const float ep = acc[t * d + i], ev = acc[t * d + N + i];
                const float np_ = r[0] * ep + (r[3] * gp_ + r[4] * gv_);          // r[3..6] = -H
                const float nv_ = r[1] * ep + r[2] * ev + (r[5] * gp_ + r[6] * gv_);
                gp_ = np_; gv_ = nv_;
                acc[t * d + i] = gp_;
                acc[t * d + N + i] = gv_;
                r[cp] += A.step * gp_;
                r[cv] += A.step * gv_;
            }
        }
        __syncthreads();
        if (last && A.grad)
            for (int k = tid; k < M; k += BS) A.grad[(size_t)bp * M + k] = acc[k];
    }
    for (int k = tid; k < M; k += BS) A.means[(size_t)bp * M + k] = rec[(k / d) * REC + REC_M + 8 + pidx(k % d)];
}

template <int N, int CHAIN, int NA, int NB>
static int launch_split_cfg(const sgpmp_shape_t& sh, const CostParams<float>& P, const IterArgs<float>& A, cudaStream_t st) {
    using Cfg = SplitCfg<NA, NB>;
    constexpr int d = 2 * N, NSTG = SPLIT_NSTG, REC = rec_floats(N);
    const int T = sh.T, M = T * d, Mpad = (M + 3) & ~3, Spad = (sh.S + 3) & ~3, NCH = (sh.S + 31) >> 5;
    const size_t phase_bytes = ((size_t)Mpad + Spad + ((NCH + 4) & ~3)) * 4;
    size_t uni = phase_bytes > Cfg::pass1_bytes() ? phase_bytes : Cfg::pass1_bytes();
    // the union region is also stg_tmp, the 32-float start / goal staging scratch of the kernel's start-up; the state-only form
    // has no pass-1 region, and with T = 2 and S <= 4 the block phases alone need only 64 or 80 bytes
    if (uni < 32 * sizeof(float)) uni = 32 * sizeof(float);
    const size_t smem = ((size_t)SPH_SMEM + (size_t)T * REC + Spad + 32 + 32) * sizeof(float) + 32 * sizeof(double) +
                        (size_t)(NB ? ((NA * (2 * NSTG + 1) + 1) & ~1) : 0) * sizeof(uint64_t) + ((uni + 15) & ~(size_t)15);
    if (smem > 227 * 1024) return SGPMP_ERR_UNSUPPORTED;
    auto kern = iterate_split_kernel<N, CHAIN, NA, NB>;
    if (smem > SGPMP_SMEM_OPTIN) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const unsigned n_cta = (unsigned)(sh.B * sh.G * sh.K);
    kern<<<n_cta, Cfg::BS, smem, st>>>(P, A);
    SGPMP_CHECK_LAUNCH("sgpmp_iterate(split)");
    return SGPMP_OK;
}

template <int CHAIN>
static int launch_split_chain(const sgpmp_shape_t& sh, const CostParams<float>& P, const IterArgs<float>& A, cudaStream_t st) {
    // equal numbers of state and link warps measured best at C4 (4,4: 14.55 ms; 4,2: 15.7; 8,4: 15.6; 4,1: 20.4; 6,2: 20.2)
    // Mid-size batches (the 4096-problem config sharded over 8 GPUs: 2,048 CTAs): 512-thread CTAs, two per SM.  The same 32 warps
    // per SM, but a CTA takes half as long, so the partial last wave costs half as much (ms per iteration, (4,4) -> (8,8):
    // 128 problems 0.529 -> 0.502, 256: 0.920 -> 0.861, 512: 1.721 -> 1.699, 1024: 3.417 -> 3.370; 4096: 13.25 -> 13.32, where
    // the finer interleave of four CTAs' block phases wins instead).
    const long n_cta = (long)sh.B * sh.G * sh.K;
    if (sh.S >= 256 && n_cta <= 6144) return launch_split_cfg<7, CHAIN, 8, 8>(sh, P, A, st);
    if (sh.S > 64) return launch_split_cfg<7, CHAIN, 4, 4>(sh, P, A, st);
    if (sh.S > 32) return launch_split_cfg<7, CHAIN, 2, 2>(sh, P, A, st);
    return launch_split_cfg<7, CHAIN, 1, 1>(sh, P, A, st);
}

// state-only form (no link fields): n_dof 2, 3, 4, 6 — the planar occupancy-map cost or no obstacle cost at all
template <int N>
static int launch_state_only(const sgpmp_shape_t& sh, const CostParams<float>& P, const IterArgs<float>& A, cudaStream_t st) {
    if (sh.S > 64) return launch_split_cfg<N, 0, 4, 0>(sh, P, A, st);
    if (sh.S > 32) return launch_split_cfg<N, 0, 2, 0>(sh, P, A, st);
    return launch_split_cfg<N, 0, 1, 0>(sh, P, A, st);
}

int launch_iterate_split(const sgpmp_shape_t& sh, const CostParams<float>& P, const IterArgs<float>& A, int chain, cudaStream_t st) {
    if (sh.T < 2) return SGPMP_ERR_UNSUPPORTED;
    if (chain == 0) {
        if (P.has_spheres || P.has_self || P.has_ee) return SGPMP_ERR_UNSUPPORTED;
        switch (sh.n_dof) {
            case 2: return launch_state_only<2>(sh, P, A, st);
            case 3: return launch_state_only<3>(sh, P, A, st);
            case 4: return launch_state_only<4>(sh, P, A, st);
            case 6: return launch_state_only<6>(sh, P, A, st);
            default: return SGPMP_ERR_UNSUPPORTED;
        }
    }
    if (sh.n_dof != 7) return SGPMP_ERR_UNSUPPORTED;
    return chain == 2 ? launch_split_chain<2>(sh, P, A, st) : launch_split_chain<1>(sh, P, A, st);
}

}  // namespace sgpmp
