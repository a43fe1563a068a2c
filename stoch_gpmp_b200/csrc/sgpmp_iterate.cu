// Fused StochGPMP optimisation loop: sample -> cost -> softmax -> weighted update, n_iters times, in
// ONE launch.  Replaces the Python loop of StochGPMP.optimize (planner.py:277-317) and everything it
// calls per iteration (sample_and_eval :239-261, _get_costs :229-237, _update_distribution :263-275).
//
// Design (B200-first, not a translation):
//   * one CTA per (problem, particle); a particle's S samples never leave the SM.  Every thread owns one
//     trajectory sample at a time and marches over t with the whole state in registers: Philox normals
//     -> banded recurrence y_t = G_t eps_t - H_t y_{t-1} -> x_t = mu_t + y_t -> cost factors/FK/obstacles.
//     No sample is written to HBM unless the caller asks for the last iteration's samples
//     (get_recent_samples, planner.py:330-337, only ever observes those).
//   * softmax over the particle's S costs in shared memory.
//   * the update uses grad = L (sum_s w_s eps_s)  (x_s - mu = L eps_s): the weighted eps-sum is
//     re-generated from the counter-based RNG with the transposed mapping thread <-> (time pair, DoF),
//     looping over s and skipping samples whose weight is exactly zero (a CTA-uniform branch: in the
//     reference's shipped configurations the softmax is one-hot, so this pass is almost free), then one
//     banded recurrence per DoF applies L.  mu and b = Sigma^-1 mu stay in shared memory across
//     iterations; particles are independent, so no grid-wide synchronisation exists anywhere.
//   * FP32-pipe/MUFU bound (DESIGN.md §6); HBM traffic is O(NP*M) per iteration instead of 3*M*S*NP.
#include <cooperative_groups.h>

#include "sgpmp_common.cuh"
#include "sgpmp_cost.cuh"
#include "sgpmp_cost_pairs.cuh"
#include "sgpmp_iterate.cuh"
#include "sgpmp_rng.cuh"

namespace cg = cooperative_groups;

namespace sgpmp {

// fp32 CTAs per SM (__launch_bounds__ minimum blocks)
constexpr int ITER_MINB256 = 3;
constexpr int ITER_MINB128 = 6;          // 6 CTAs x 4 warps at 80 registers: the same 24 warps/SM as 3 x 256 threads, finer block phases
constexpr int ITER_MINB128_SMALL = 10;   // n_dof <= 3 (planar): the whole state is 4-6 registers; 51 registers per thread, 10 CTAs per SM (8: 1.79 ms, 10: 1.77, 12: 1.81)

// PACK selects the pass-1 arithmetic:
//   0  scalar: one sample per thread (fp32 or fp64)
//   2  one fp32 sample per thread, packed arithmetic across neighbouring DoFs / links (sgpmp_cost_pairs.cuh)
// CL > 1: one particle's S samples are split over a thread-block CLUSTER of CL CTAs (low-latency mode for few
// problems: B*NP CTAs cannot fill 148 SMs).  Each CTA draws and scores samples [cr*S/CL, (cr+1)*S/CL) with the same
// global RNG counters; the softmax statistics (max, sum) and the weighted eps-sum are exchanged through distributed
// shared memory (cluster.map_shared_rank) with four cluster barriers per iteration, then every CTA applies the
// identical update to its own copy of mu.  No global memory or extra launch is involved.
template <typename real, int PACK, int N, int BS, int CHAIN, int CL>
__global__ void __launch_bounds__(BS, (sizeof(real) == 4 ? (BS == 256 ? ITER_MINB256 : ((N <= 3 && CL == 1 && BS == 128) ? ITER_MINB128_SMALL : ITER_MINB128)) : 1))
iterate_kernel(const __grid_constant__ CostParams<real> P, const __grid_constant__ IterArgs<real> A) {
    constexpr int d = 2 * N;
    constexpr int NP2 = (N + 1) / 2;
    constexpr int VOFF = (PACK == 2) ? 2 * NP2 : N;                   // offset of the velocity half in a shared-memory row
    constexpr int DP = (PACK == 2) ? 2 * VOFF : ((d + 3) & ~3);       // padded row length of mu / b (16-byte aligned rows)
    auto col = [](int j) { return j < N ? j : VOFF + (j - N); };      // external state index -> shared-memory column
    const int T = A.T, S = A.S, G = A.G, K = A.K;
    const int M = T * d;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    real* sph = reinterpret_cast<real*>(smem_raw);            // [MAX_SPHERES][8] + coll_const (16-byte aligned)
    real* tabGH = sph + SPH_SMEM;                             // [T][8]  (g11 g21 g22 h11 | h12 h21 h22 -)
    real* mu = tabGH + (size_t)T * 8;                         // [T][DP]
    real* bvec = mu + (size_t)T * DP;                         // [T][DP]
    double* tabDO = reinterpret_cast<double*>(bvec + (size_t)T * DP);   // [T][7]
    double* red64 = tabDO + (size_t)T * 7;                              // [32] fp64 reduction scratch
    real* acc = reinterpret_cast<real*>(red64 + 32);                    // [T][d]  sum_s w_s eps_s, then grad
    real* wsm = acc + M;                                      // [ceil(S/CL)] costs -> weights of this CTA's samples
    real* part = wsm + (S + CL - 1) / CL;                     // [4*BS] partial sums of pass 2
    real* red = part + 4 * BS;                                // [32]
    real* start = red + 32;                                   // [2*VOFF]
    real* goal = start + 2 * VOFF;                            // [2*VOFF]
    real* xch = goal + 2 * VOFF;                              // [4]   cluster exchange: local max, local sum
    real* accsum = xch + 4;                                   // [T][d] cluster-reduced eps-sum (CL > 1 only)

    const int NP = G * K;
    const int bp = blockIdx.x / CL, cr = blockIdx.x % CL, b = bp / NP, p = bp - b * NP;
    const int n_particles = gridDim.x / CL;
    const int S_loc = (S + CL - 1) / CL;
    const int s_lo = cr * S_loc, s_hi = min(S, s_lo + S_loc), ns = max(0, s_hi - s_lo);   // this CTA's samples
    const int tid = threadIdx.x;
    const uint32_t pgid = A.particle_gid0 + (uint32_t)bp;

    for (int k = tid; k < T * 8; k += BS) {
        const int t = k >> 3, c = k & 7;
        const double* row = A.tab + (size_t)t * SGPMP_TABLE_STRIDE;
        tabGH[k] = c < 7 ? (real)row[c] : (real)0;
        if (c < 7) tabDO[t * 7 + c] = row[SGPMP_TAB_D11 + c];
    }
    for (int k = tid; k < T * DP; k += BS) { mu[k] = 0; bvec[k] = 0; }
    __syncthreads();
    for (int k = tid; k < M; k += BS) mu[(k / d) * DP + col(k % d)] = A.means[(size_t)bp * M + k];
    stage_cta_constants<real, N, CHAIN, VOFF>(P, b, p / K, G, start, goal, sph);
    CostSmem<real> sm;
    sm.start = start; sm.goal = goal; sm.bvec = bvec; sm.sph = sph;
    sm.coll_const = sph[SPH_STRIDE * SGPMP_MAX_SPHERES];
    sm.self_const = sph[SPH_STRIDE * SGPMP_MAX_SPHERES + 1];
    sm.map = P.has_map ? P.occ_map + (size_t)(P.map_of_problem ? P.map_of_problem[b] : 0) * P.map_h * P.map_w : nullptr;
    sm.map_u8 = (P.has_map && P.occ_map_u8) ? P.occ_map_u8 + (size_t)(P.map_of_problem ? P.map_of_problem[b] : 0) * P.map_h * P.map_w : nullptr;
    __syncthreads();

    for (int it = 0; it < A.n_iters; ++it) {
        const bool last = (it == A.n_iters - 1);
        const RngKey& key = A.key;
        const uint32_t dro = (uint32_t)it;      // draw index of this iteration = key.draw + it
        const real* eps = A.eps_in ? A.eps_in + ((size_t)it * n_particles + bp) * (size_t)M * S : nullptr;

        // ---- b = Sigma^-1 mu (fp64 accumulate) ---------------------------------------------------------
        double mub_part = 0.0;
        for (int k = tid; k < T * N; k += BS) {
            const int t = k / N, i = k - t * N;
            mub_part += precision_times_row<real, DP, VOFF>(tabDO, mu, T, N, t, i, &bvec[t * DP + i], &bvec[t * DP + VOFF + i]);
        }
        sm.mub = (real)block_sum_f64(mub_part, red64);
        if (last && A.means_pre && cr == 0)
            for (int k = tid; k < M; k += BS) A.means_pre[(size_t)bp * M + k] = mu[(k / d) * DP + col(k % d)];
        __syncthreads();

        // ---- pass 1: sample + cost, one thread per trajectory sample -----------------------------------
        const bool emit = last && A.samples != nullptr;
        if constexpr (PACK == 2) {
            // one sample per thread, DoF pairs packed (sgpmp_cost_pairs.cuh)
            for (int s0 = s_lo + tid; s0 < s_hi; s0 += BS) {
                TrajCostPairs<N, CHAIN> tc;
                tc.begin();
                F2 yp[NP2], yv[NP2];
#pragma unroll
                for (int k = 0; k < NP2; ++k) yp[k] = yv[k] = f2(0.f, 0.f);
#pragma unroll 1                        // 2 was measured slower (DESIGN.md §6)
                for (int t = 0; t < T; ++t) {
                    F2 ep[NP2], ev[NP2];
                    if (eps) {
#pragma unroll
                        for (int k = 0; k < NP2; ++k) {
                            const int i0 = 2 * k, i1 = 2 * k + 1;
                            const real* r0 = eps + ((size_t)t * d) * S + s0;
                            ep[k] = f2(r0[(size_t)i0 * S], i1 < N ? r0[(size_t)i1 * S] : 0.f);
                            ev[k] = f2(r0[(size_t)(N + i0) * S], i1 < N ? r0[(size_t)(N + i1) * S] : 0.f);
                        }
                    } else {
#pragma unroll
                        for (int k = 0; k < NP2; ++k) {
                            if (2 * k + 1 < N) normal_pair_f2<true>(key, (uint32_t)t, (uint32_t)k, A.sample_gid0 + (uint32_t)s0, pgid, ep[k], ev[k], dro);
                            else normal_pair_f2<false>(key, (uint32_t)t, (uint32_t)k, A.sample_gid0 + (uint32_t)s0, pgid, ep[k], ev[k], dro);
                        }
                    }
                    real r[8];
                    load4(tabGH + t * 8, r[0], r[1], r[2], r[3]);
                    load4(tabGH + t * 8 + 4, r[4], r[5], r[6], r[7]);
                    const real* mrow = mu + t * DP;
                    F2 xp[NP2], xv[NP2];
#pragma unroll
                    for (int k = 0; k < NP2; ++k) {
                        const F2 np_ = vfma(r[0], ep[k], vneg(vfma(r[3], yp[k], r[4] * yv[k])));
                        const F2 nv_ = vfma(r[1], ep[k], r[2] * ev[k]) - vfma(r[5], yp[k], r[6] * yv[k]);
                        yp[k] = np_; yv[k] = nv_;
                        xp[k] = f2(mrow[2 * k], mrow[2 * k + 1]) + np_;
                        xv[k] = f2(mrow[VOFF + 2 * k], mrow[VOFF + 2 * k + 1]) + nv_;
                    }
                    tc.step(P, sm, t, T, xp, xv, yp, yv, bvec + t * DP);
                    if (emit) {
#pragma unroll
                        for (int k = 0; k < NP2; ++k) {
                            real* row = A.samples + ((size_t)bp * M + (size_t)t * d) * S + s0;
                            row[(size_t)(2 * k) * S] = lane0(xp[k]);
                            row[(size_t)(N + 2 * k) * S] = lane0(xv[k]);
                            if (2 * k + 1 < N) { row[(size_t)(2 * k + 1) * S] = lane1(xp[k]); row[(size_t)(N + 2 * k + 1) * S] = lane1(xv[k]); }
                        }
                    }
                }
                const real c = tc.total(P, sm, T, nullptr);
                wsm[s0 - s_lo] = c;
                if (last && A.costs) A.costs[(size_t)bp * S + s0] = c;
            }
        } else {
            for (int s0 = s_lo + tid; s0 < s_hi; s0 += BS) {
                TrajCost<real, N, CHAIN> tc;
                tc.begin();
                real yp[N], yv[N];
    #pragma unroll
                for (int i = 0; i < N; ++i) { yp[i] = 0; yv[i] = 0; }
                // One Philox call yields the four normals of a DoF pair; the step body is kept as a
                // single (not 2x unrolled) copy so that the hot loop stays inside the instruction cache.
    #pragma unroll 1
                for (int t = 0; t < T; ++t) {
                    real e[d + 1];
                    if (eps) {
    #pragma unroll
                        for (int j = 0; j < d; ++j) {
                            const real* row = eps + ((size_t)t * d + j) * S;
                            e[j] = row[s0];
                        }
                    } else {
    #pragma unroll
                        for (int k = 0; k < (N + 1) / 2; ++k) {
                            const bool full = (2 * k + 1 < N);
                            real p1, v1;
                            normal_pair<real>(key, (uint32_t)t, (uint32_t)k, full, A.sample_gid0 + (uint32_t)s0, pgid, e[2 * k], p1, e[N + 2 * k], v1, dro);
                            if (full) { e[2 * k + 1] = p1; e[N + 2 * k + 1] = v1; }
                        }
                    }
                    real r[8], m[DP];
                    load4(tabGH + t * 8, r[0], r[1], r[2], r[3]);
                    load4(tabGH + t * 8 + 4, r[4], r[5], r[6], r[7]);
    #pragma unroll
                    for (int q = 0; q < DP / 4; ++q) load4(mu + t * DP + 4 * q, m[4 * q], m[4 * q + 1], m[4 * q + 2], m[4 * q + 3]);
                    real x[d];
    #pragma unroll
                    for (int i = 0; i < N; ++i) {
                        const real np_ = vfma(r[0], e[i], vneg(vfma(r[3], yp[i], r[4] * yv[i])));
                        const real nv_ = vfma(r[1], e[i], r[2] * e[N + i]) - vfma(r[5], yp[i], r[6] * yv[i]);
                        yp[i] = np_; yv[i] = nv_;
                        x[i] = m[i] + np_;
                        x[N + i] = m[N + i] + nv_;
                    }
                    tc.step(P, sm, t, T, x, yp, yv, bvec + t * DP);
                    if (emit) {
    #pragma unroll
                        for (int j = 0; j < d; ++j) {
                            real* row = A.samples + ((size_t)bp * M + (size_t)t * d + j) * S;
                            row[s0] = x[j];
                        }
                    }
                }
                tc.finish(P, sm, T);
                const real c = tc.total();
                wsm[s0 - s_lo] = c;
                if (last && A.costs) A.costs[(size_t)bp * S + s0] = c;
            }
        }
        __syncthreads();

        // ---- softmax over the S samples of this particle (cluster-wide when CL > 1) ----------------------
        {
            real m = -INFINITY;
            for (int s = tid; s < ns; s += BS) {
                const real z = -wsm[s] / P.temperature;
                wsm[s] = z;
                m = sg_max(m, z);
            }
            m = warp_max(m);
            if ((tid & 31) == 0) red[tid >> 5] = m;
            __syncthreads();
            m = red[0];
            for (int k = 1; k < BS / 32; ++k) m = sg_max(m, red[k]);
            if constexpr (CL > 1) {
                cg::cluster_group cluster = cg::this_cluster();
                if (tid == 0) xch[0] = m;
                cluster.sync();
                for (int r = 0; r < CL; ++r) m = sg_max(m, *cluster.map_shared_rank(xch, r));
            }
            __syncthreads();
            real Z = 0;
            for (int s = tid; s < ns; s += BS) {
                const real ex = sg_exp(wsm[s] - m);
                wsm[s] = ex;
                Z += ex;
            }
            Z = warp_sum(Z);
            if ((tid & 31) == 0) red[tid >> 5] = Z;
            __syncthreads();
            Z = 0;
            for (int k = 0; k < BS / 32; ++k) Z += red[k];
            if constexpr (CL > 1) {
                cg::cluster_group cluster = cg::this_cluster();
                if (tid == 0) xch[1] = Z;
                cluster.sync();
                Z = 0;
                for (int r = 0; r < CL; ++r) Z += *cluster.map_shared_rank(xch + 1, r);     // fixed rank order: identical on every CTA
            }
            if (A.stats_out) {
                // split-particle mode: the weights stay UNNORMALISED (exp(z - m) of this rank's samples); (m, Z) go out with A
                if (tid == 0) { A.stats_out[(size_t)bp * (M + 2)] = m; A.stats_out[(size_t)bp * (M + 2) + 1] = Z; }
            } else {
                for (int s = tid; s < ns; s += BS) {
                    const real w = wsm[s] / Z;
                    wsm[s] = w;
                    if (last && A.weights) A.weights[(size_t)bp * S + s_lo + s] = w;
                }
            }
            __syncthreads();
        }

        // ---- pass 2: acc = sum_s w_s eps_s --------------------------------------------------------------
        if (eps) {
            const int warp = tid >> 5, lane = tid & 31;
            for (int r = warp; r < M; r += BS / 32) {
                real a = 0;
                for (int s = lane; s < ns; s += 32) a += wsm[s] * eps[(size_t)r * S + s_lo + s];
                a = warp_sum(a);
                if (lane == 0) acc[r] = a;
            }
        } else {
            constexpr int NPAIR = (N + 1) / 2;
            const int n_items = T * NPAIR;                    // one item = the 4 normals of (time step, DoF pair)
            const int nsplit = (n_items < BS) ? (BS / n_items) : 1;
            for (int base = 0; base < n_items; base += BS) {
                const int item = base + (tid % (nsplit > 1 ? n_items : BS));
                const int split = (nsplit > 1) ? tid / n_items : 0;
                const bool active = item < n_items && split < nsplit;
                real a0 = 0, a1 = 0, a2 = 0, a3 = 0;
                const int t_ = item / NPAIR, k = item - t_ * NPAIR;
                const bool full = (2 * k + 1 < N);
                if (active) {
                    for (int s = split; s < ns; s += nsplit) {
                        const real w = wsm[s];
                        if (w == (real)0) continue;
                        real p0, p1, v0, v1;
                        normal_pair<real>(key, (uint32_t)t_, (uint32_t)k, full, A.sample_gid0 + (uint32_t)(s_lo + s), pgid, p0, p1, v0, v1, dro);
                        a0 += w * p0; a1 += w * p1; a2 += w * v0; a3 += w * v1;
                    }
                }
                if (nsplit > 1) {
                    part[4 * tid + 0] = a0; part[4 * tid + 1] = a1; part[4 * tid + 2] = a2; part[4 * tid + 3] = a3;
                    __syncthreads();
                    if (active && split == 0) {
                        for (int q = 1; q < nsplit; ++q) {
                            const real* pp = part + 4 * (q * n_items + item);
                            a0 += pp[0]; a1 += pp[1]; a2 += pp[2]; a3 += pp[3];
                        }
                    }
                }
                if (active && split == 0) {
                    acc[t_ * d + 2 * k] = a0;
                    acc[t_ * d + N + 2 * k] = a2;
                    if (full) {
                        acc[t_ * d + 2 * k + 1] = a1;
                        acc[t_ * d + N + 2 * k + 1] = a3;
                    }
                }
            }
        }
        __syncthreads();
        if constexpr (CL > 1) {
            // all-reduce of the partial eps-sums over the cluster through distributed shared memory
            cg::cluster_group cluster = cg::this_cluster();
            cluster.sync();
            for (int k = tid; k < M; k += BS) {
                real a = 0;
                for (int r = 0; r < CL; ++r) a += cluster.map_shared_rank(acc, r)[k];
                accsum[k] = a;
            }
            cluster.sync();                       // every CTA has read every partial before acc is reused
            for (int k = tid; k < M; k += BS) acc[k] = accsum[k];
            __syncthreads();
        }

        if (A.stats_out) {       // split-particle mode: hand A = sum_s exp(z_s - m) eps_s to the exchange, no update here
            for (int k = tid; k < M; k += BS) A.stats_out[(size_t)bp * (M + 2) + 2 + k] = acc[k];
            return;
        }
        // ---- grad = L acc (banded recurrence, one thread per DoF); mu += step * grad --------------------
        if (tid < N) {
            const int i = tid;
            real gp_ = 0, gv_ = 0;
            for (int t = 0; t < T; ++t) {
                const real* r = tabGH + t * 8;
                const real ep = acc[t * d + i], ev = acc[t * d + N + i];
                const real np_ = r[0] * ep - (r[3] * gp_ + r[4] * gv_);
                const real nv_ = r[1] * ep + r[2] * ev - (r[5] * gp_ + r[6] * gv_);
                gp_ = np_; gv_ = nv_;
                acc[t * d + i] = gp_;
                acc[t * d + N + i] = gv_;
                mu[t * DP + i] += A.step * gp_;
                mu[t * DP + VOFF + i] += A.step * gv_;
            }
        }
        __syncthreads();
        if (last && A.grad && cr == 0)
            for (int k = tid; k < M; k += BS) A.grad[(size_t)bp * M + k] = acc[k];
    }
    if (cr == 0)
        for (int k = tid; k < M; k += BS) A.means[(size_t)bp * M + k] = mu[(k / d) * DP + col(k % d)];
}

template <typename real, int PACK, int N, int BS, int CHAIN, int CL = 1>
static int launch_iterate_nb(const sgpmp_shape_t& sh, const CostParams<real>& P, const IterArgs<real>& A, cudaStream_t st) {
    const int d = 2 * N, M = sh.T * d, VOFF = (PACK == 2) ? 2 * ((N + 1) / 2) : N, DP = (PACK == 2) ? 2 * VOFF : ((d + 3) & ~3);
    const int S_loc = (sh.S + CL - 1) / CL;
    const size_t smem = ((size_t)sh.T * 7 + 32) * sizeof(double) +
                        ((size_t)sh.T * (8 + 2 * DP) + (size_t)M * (CL > 1 ? 2 : 1) + S_loc + 4 * BS + 32 + 4 * VOFF + 4 + SPH_SMEM) * sizeof(real);
    if (smem > 227 * 1024) {
        set_error("sgpmp_iterate: T=%d, S=%d need %zu bytes of shared memory (> 227 KiB)", sh.T, sh.S, smem);
        return SGPMP_ERR_UNSUPPORTED;
    }
    auto kern = iterate_kernel<real, PACK, N, BS, CHAIN, CL>;
    if (smem > SGPMP_SMEM_OPTIN) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const unsigned n_cta = (unsigned)(sh.B * sh.G * sh.K) * CL;
    if constexpr (CL > 1) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(n_cta);
        cfg.blockDim = dim3(BS);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = CL;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        cudaLaunchKernelEx(&cfg, kern, P, A);
    } else {
        kern<<<n_cta, BS, smem, st>>>(P, A);
    }
    SGPMP_CHECK_LAUNCH("sgpmp_iterate");
    return SGPMP_OK;
}

// few problems: split every particle's samples over a cluster of 8 / 4 / 2 CTAs (DSMEM reductions) so that the
// launch still covers the 148 SMs: the largest cluster that keeps <= 2 CTAs per SM and >= 64 samples per CTA
static int iterate_cluster_size(const sgpmp_shape_t& sh, bool injected_eps) {
    const long n_part = (long)sh.B * sh.G * sh.K;
    if (injected_eps) return 1;
    for (int c = 8; c >= 2; c >>= 1)
        if (n_part * c <= 2 * 148 && sh.S >= 64 * c && (c == 8 ? sh.S >= 256 : true)) return c;
    return 1;
}

// fp32 dof-pair pass 1 (PACK 2): the Panda structure (CHAIN 1, 2) and, with CHAIN 0, costs without link fields (occupancy map or
// no obstacle cost).  Cluster mode for few problems.
template <int N, int CHAIN>
static int launch_iterate_pairs(const sgpmp_shape_t& sh, const CostParams<float>& P, const IterArgs<float>& A, cudaStream_t st) {
    const int cl = A.stats_out ? 1 : iterate_cluster_size(sh, A.eps_in != nullptr);
    if (cl == 8) return launch_iterate_nb<float, 2, N, 64, CHAIN, 8>(sh, P, A, st);
    if (cl == 4) return launch_iterate_nb<float, 2, N, 128, CHAIN, 4>(sh, P, A, st);
    if (cl == 2) return launch_iterate_nb<float, 2, N, 128, CHAIN, 2>(sh, P, A, st);
    // CTA size.  Chains with link fields (Panda): 256 threads, 3 CTAs/SM.  (128 threads at 6 CTAs/SM — the same 24 warps per SM —
    // measured 17.19 against 17.41 ms at 4096 problems, but 1.65 against 1.20 ms at 256 problems and 4.80 against 4.56 ms at 1024:
    // each CTA then runs twice as long, so the last partial wave costs more than the finer block phases gain.)  Without link fields
    // (planar: a short per-sample body, so the per-iteration block phases — b = P mu, softmax, update — weigh more and 80 registers
    // are not needed) 128-thread CTAs at 10 CTAs/SM and 48 registers give 2.23 -> 1.81 ms at 4096 x 4 x 256; grids too small to
    // fill that keep 256 threads.
    const long n_part = (long)sh.B * sh.G * sh.K;
    const bool light = (CHAIN == 0) && !(P.has_spheres || P.has_self);
    if (sh.S > 128 && !(light && n_part >= 10L * 148)) return launch_iterate_nb<float, 2, N, 256, CHAIN>(sh, P, A, st);
    return launch_iterate_nb<float, 2, N, 128, CHAIN>(sh, P, A, st);
}

// every cost list without the Panda structure: dof pairs where they apply, else the scalar pass 1 (fp64, generic FK chains,
// the other DoF counts)
template <typename real, int N>
static int launch_iterate_n(const sgpmp_shape_t& sh, const CostParams<real>& P, const IterArgs<real>& A, cudaStream_t st) {
    if constexpr (sizeof(real) == 4 && (N == 2 || N == 7)) {
        if (!(P.has_spheres || P.has_self)) return launch_iterate_pairs<N, 0>(sh, P, A, st);
    }
    if (sh.S > 128) return launch_iterate_nb<real, 0, N, 256, 0>(sh, P, A, st);
    return launch_iterate_nb<real, 0, N, 128, 0>(sh, P, A, st);
}

template <typename real>
static int launch_iterate(const sgpmp_shape_t& sh, const sgpmp_cost_desc_t& desc, const double* tables, double step,
                          int n_iters, const void* eps_in, uint64_t seed, uint32_t draw0, void* means, void* means_pre,
                          void* samples, void* costs, void* weights, void* grad, cudaStream_t st, void* stats_out = nullptr) {
    CostParams<real> P;
    int rc = lower_cost_desc<real>(sh, desc, P);
    if (rc != SGPMP_OK) return rc;
    if (!(desc.temperature > 0)) { set_error("sgpmp_iterate: temperature must be > 0"); return SGPMP_ERR_INVALID_ARG; }
    IterArgs<real> A;
    A.G = sh.G; A.K = sh.K; A.S = sh.S; A.T = sh.T; A.n_iters = n_iters;
    A.particle_gid0 = (uint32_t)(sh.problem_gid0 * sh.G * sh.K);
    A.sample_gid0 = (uint32_t)sh.sample_gid0;
    A.step = (real)step;
    A.key = make_rng_key(seed, draw0);
    A.tab = tables;
    A.eps_in = (const real*)eps_in;
    A.means = (real*)means; A.means_pre = (real*)means_pre; A.samples = (real*)samples;
    A.costs = (real*)costs; A.weights = (real*)weights; A.grad = (real*)grad;
    A.stats_out = (real*)stats_out;
    if constexpr (sizeof(real) == 4) {
        // the role-split kernel (sgpmp_iterate_split.cu) unless the grid is small enough for cluster mode; the single-role
        // kernel also takes the shapes it does not support (T < 2, shared memory beyond 227 KiB at large S)
        const bool split = A.stats_out || iterate_cluster_size(sh, A.eps_in != nullptr) == 1;
        if (structured_fields_ok(P) && chain_is_panda_structure(desc, sh.n_dof)) {
            if (split) {
                rc = launch_iterate_split(sh, P, A, P.has_self ? 2 : 1, st);
                if (rc != SGPMP_ERR_UNSUPPORTED) return rc;
            }
            return P.has_self ? launch_iterate_pairs<7, 2>(sh, P, A, st) : launch_iterate_pairs<7, 1>(sh, P, A, st);
        }
        // no link fields (planar occupancy map / no obstacle cost): the state-only form of the record-layout kernel
        if (split && !(P.has_spheres || P.has_self || P.has_ee)) {
            rc = launch_iterate_split(sh, P, A, 0, st);
            if (rc != SGPMP_ERR_UNSUPPORTED) return rc;
        }
    }
    switch (sh.n_dof) {
#define SGPMP_DOF_CASE(N) case N: return launch_iterate_n<real, N>(sh, P, A, st);
#include "sgpmp_dof_list.inc"
#undef SGPMP_DOF_CASE
        default:
            set_error("sgpmp_iterate: n_dof=%d is not instantiated (see sgpmp_dof_list.inc)", sh.n_dof);
            return SGPMP_ERR_UNSUPPORTED;
    }
}

int iterate_stats_launch(const sgpmp_shape_t& sh, const sgpmp_cost_desc_t& desc, const double* tables, uint64_t seed,
                         uint32_t draw, const void* means, void* costs, void* stats, cudaStream_t st) {
    // one pass of sample -> cost -> local softmax statistics over THIS launch's samples (sample_gid0 .. + S); means are read only
    if (sh.dtype == SGPMP_F32)
        return launch_iterate<float>(sh, desc, tables, 0.0, 1, nullptr, seed, draw, const_cast<void*>(means), nullptr, nullptr, costs,
                                     nullptr, nullptr, st, stats);
    return launch_iterate<double>(sh, desc, tables, 0.0, 1, nullptr, seed, draw, const_cast<void*>(means), nullptr, nullptr, costs,
                                  nullptr, nullptr, st, stats);
}

}  // namespace sgpmp

using namespace sgpmp;

extern "C" int sgpmp_iterate_stats(const sgpmp_shape_t* shape, const sgpmp_cost_desc_t* desc, const double* tables,
                                   uint64_t seed, uint32_t draw, const void* means, void* costs, void* stats, void* stream) {
    SGPMP_REQUIRE(shape_ok(shape), "sgpmp_iterate_stats: invalid shape");
    SGPMP_REQUIRE(desc && tables && means && stats, "sgpmp_iterate_stats: null pointer");
    return iterate_stats_launch(*shape, *desc, tables, seed, draw, means, costs, stats, (cudaStream_t)stream);
}

extern "C" int sgpmp_iterate(const sgpmp_shape_t* shape, const sgpmp_cost_desc_t* desc, const double* tables,
                             double step_size, int32_t n_iters, const void* eps_in, uint64_t seed, uint32_t draw0,
                             void* means, void* means_pre, void* samples, void* costs, void* weights, void* grad,
                             void* stream) {
    SGPMP_REQUIRE(shape_ok(shape), "sgpmp_iterate: invalid shape");
    SGPMP_REQUIRE(desc && tables && means, "sgpmp_iterate: null pointer");
    SGPMP_REQUIRE(n_iters >= 1, "sgpmp_iterate: n_iters must be >= 1");
    if (shape->dtype == SGPMP_F32)
        return launch_iterate<float>(*shape, *desc, tables, step_size, n_iters, eps_in, seed, draw0, means, means_pre,
                                     samples, costs, weights, grad, (cudaStream_t)stream);
    return launch_iterate<double>(*shape, *desc, tables, step_size, n_iters, eps_in, seed, draw0, means, means_pre,
                                  samples, costs, weights, grad, (cudaStream_t)stream);
}
