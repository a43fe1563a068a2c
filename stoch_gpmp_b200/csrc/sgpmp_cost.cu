// K3 — standalone per-trajectory-sample cost kernel, and the host-side lowering of sgpmp_cost_desc_t.
// (Arithmetic and reference citations: sgpmp_cost.cuh.)
//
// Mapping: one thread per trajectory sample marching over t; the S-minor sample layout makes the 2n
// loads of a step fully coalesced across the warp.  Per-particle constants (start, goal, b = P mu,
// sphere table) are staged in shared memory once per CTA.
#include <math.h>

#include "sgpmp_common.cuh"
#include "sgpmp_cost.cuh"

namespace sgpmp {

template <typename real>
int lower_cost_desc(const sgpmp_shape_t& sh, const sgpmp_cost_desc_t& d, CostParams<real>& o) {
    memset(&o, 0, sizeof(o));
    if (!(d.dt > 0) || !(d.sigma_gp > 0) || !d.start) {
        set_error("cost desc: dt, sigma_gp must be > 0 and start non-null");
        return SGPMP_ERR_INVALID_ARG;
    }
    o.dt = (real)d.dt;
    // sigma_start <= 0: no start factor (CostGPTrajectory, cost_functions.py:171-218: the GP transition factors alone)
    o.inv_sig_start2 = d.sigma_start > 0 ? (real)(1.0 / (d.sigma_start * d.sigma_start)) : (real)0;
    // Q^-1 blocks exactly as GPFactor.calc_Q_inv forms them (gp_factor.py:44-52)
    const double qc = 1.0 / (d.sigma_gp * d.sigma_gp);
    o.q11 = (real)(12.0 * pow(d.dt, -3.0) * qc);
    o.q12x2 = (real)(2.0 * (-6.0 * pow(d.dt, -2.0) * qc));
    o.q22 = (real)(4.0 * pow(d.dt, -1.0) * qc);
    o.temperature = (real)d.temperature;
    o.start = (const real*)d.start;
    o.goals = (const real*)d.goals;
    o.has_goal = (d.goals != nullptr && d.sigma_goal_prior > 0) ? 1 : 0;
    o.inv_sig_goal2 = o.has_goal ? (real)(1.0 / (d.sigma_goal_prior * d.sigma_goal_prior)) : (real)0;
    o.has_map = d.occ_map != nullptr;
    o.has_spheres = d.spheres != nullptr && d.n_spheres > 0;
    if (o.has_map) {
        if (d.map_h <= 0 || d.map_w <= 0 || d.n_maps <= 0 || !(d.map_sigma_coll > 0)) {
            set_error("cost desc: bad occupancy-map parameters");
            return SGPMP_ERR_INVALID_ARG;
        }
        if (d.map_h != d.map_w) {
            set_error("cost desc: non-square occupancy maps are not supported (the reference's clamp "
                      "obst_map.py:177-178 is only well defined for square maps)");
            return SGPMP_ERR_UNSUPPORTED;
        }
        if (sh.n_dof < 2) { set_error("cost desc: occupancy map needs n_dof >= 2"); return SGPMP_ERR_INVALID_ARG; }
        o.occ_map = (const real*)d.occ_map;
        o.occ_map_u8 = d.occ_map_u8;
        o.map_of_problem = d.map_of_problem;
        o.map_h = d.map_h; o.map_w = d.map_w; o.n_maps = d.n_maps;
        o.origin_xi = d.origin_xi; o.origin_yi = d.origin_yi;
        o.map_inv_cell = (real)d.map_inv_cell;
        o.map_origin_x = (real)d.origin_xi;
        o.map_origin_y = (real)d.origin_yi;
        o.map_w_coll = (real)(1.0 / (d.map_sigma_coll * d.map_sigma_coll));
    }
    o.has_self = d.self_margin > 0;
    if (o.has_self && !(d.self_sigma_coll > 0)) { set_error("cost desc: self_sigma_coll must be > 0"); return SGPMP_ERR_INVALID_ARG; }
    if (o.has_spheres && (d.n_spheres > SGPMP_MAX_SPHERES || !(d.sphere_sigma_coll > 0))) {
        set_error("cost desc: n_spheres must be <= %d and sigma_coll > 0", SGPMP_MAX_SPHERES);
        return SGPMP_ERR_INVALID_ARG;
    }
    o.has_ee = d.ee_sigma_goal > 0;
    if (o.has_spheres || o.has_self || o.has_ee) {
        if (o.has_map) { set_error("cost desc: link fields and an occupancy map cannot be combined"); return SGPMP_ERR_UNSUPPORTED; }
        if (d.n_frames < sh.n_dof || d.n_frames > SGPMP_MAX_FRAMES) {
            set_error("cost desc: FK chain needs n_dof <= n_frames <= %d", SGPMP_MAX_FRAMES);
            return SGPMP_ERR_INVALID_ARG;
        }
        for (int f = 0; f < d.n_frames; ++f) {
            const int want = f < sh.n_dof ? f : -1;
            if (d.chain_joint[f] != want) {
                set_error("cost desc: FK chain must be a serial arm: frames 0..n_dof-1 revolute-z with joint f, "
                          "then fixed frames (frame %d has joint %d)", f, d.chain_joint[f]);
                return SGPMP_ERR_UNSUPPORTED;
            }
        }
        o.n_frames = d.n_frames;
        o.include_base = d.include_base;
        for (int f = 0; f < d.n_frames; ++f) {
            for (int k = 0; k < 9; ++k) o.R[f][k] = (real)d.chain_R[f][k];
            for (int k = 0; k < 3; ++k) o.p[f][k] = (real)d.chain_p[f][k];
            o.joint[f] = d.chain_joint[f];
        }
    }
    if (o.has_spheres) {
        o.spheres = (const real*)d.spheres;
        o.n_spheres = d.n_spheres;
        o.spheres_per_problem = d.spheres_per_problem;
        if (d.sphere_field_type < SGPMP_FIELD_RBF || d.sphere_field_type > SGPMP_FIELD_OCCUPANCY) {
            set_error("cost desc: unknown sphere_field_type %d", d.sphere_field_type);
            return SGPMP_ERR_INVALID_ARG;
        }
        o.sphere_mode = d.sphere_field_type;
        o.sphere_w_coll = (real)(1.0 / (d.sphere_sigma_coll * d.sphere_sigma_coll));
    }
    if (o.has_self) {
        o.self_k = (real)((sizeof(real) == 4 ? -0.5 * 1.4426950408889634 : -0.5) / (d.self_margin * d.self_margin));
        o.self_w_coll = (real)(1.0 / (d.self_sigma_coll * d.self_sigma_coll));
    }
    // link interpolation: indices address the link list (base first when include_base)
    const int L = d.n_frames + (d.include_base ? 1 : 0);
    auto interp_ok = [&](int n, int lo, int hi, const char* which) {
        if (n == 0) return true;
        if (n < 0 || n > SGPMP_MAX_INTERP || lo < 0 || hi < lo || hi > L - 1 || L + n * (hi - lo) > SGPMP_MAX_LINK_POINTS) {
            set_error("cost desc: %s interpolation needs 0 <= n <= %d, 0 <= lo <= hi <= L-1 = %d and at most %d points "
                      "(n=%d, range [%d,%d))", which, SGPMP_MAX_INTERP, L - 1, SGPMP_MAX_LINK_POINTS, n, lo, hi);
            return false;
        }
        return true;
    };
    if (o.has_spheres) {
        if (!interp_ok(d.sphere_interp_n, d.sphere_interp_lo, d.sphere_interp_hi, "sphere-field")) return SGPMP_ERR_INVALID_ARG;
        o.sphere_interp_n = d.sphere_interp_n; o.sphere_interp_lo = d.sphere_interp_lo; o.sphere_interp_hi = d.sphere_interp_hi;
        for (int k = 0; k < d.sphere_interp_n; ++k) o.sphere_alpha[k] = (real)d.sphere_interp_alpha[k];
    }
    if (o.has_self) {
        if (!interp_ok(d.self_interp_n, d.self_interp_lo, d.self_interp_hi, "self-field")) return SGPMP_ERR_INVALID_ARG;
        o.self_interp_n = d.self_interp_n; o.self_interp_lo = d.self_interp_lo; o.self_interp_hi = d.self_interp_hi;
        for (int k = 0; k < d.self_interp_n; ++k) o.self_alpha[k] = (real)d.self_interp_alpha[k];
    }
    if (o.has_ee) {
        if (!(d.ee_w_pos >= 0) || !(d.ee_w_rot >= 0)) { set_error("cost desc: ee_w_pos / ee_w_rot must be >= 0"); return SGPMP_ERR_INVALID_ARG; }
        for (int k = 0; k < 9; ++k) o.ee_R[k] = (real)d.ee_target_R[k];
        for (int k = 0; k < 3; ++k) o.ee_p[k] = (real)d.ee_target_p[k];
        o.ee_w_pos = (real)d.ee_w_pos; o.ee_w_rot = (real)d.ee_w_rot;
        o.ee_w = (real)(1.0 / (d.ee_sigma_goal * d.ee_sigma_goal));
        o.ee_square = d.ee_square ? 1 : 0;
    }
    return SGPMP_OK;
}
template int lower_cost_desc<float>(const sgpmp_shape_t&, const sgpmp_cost_desc_t&, CostParams<float>&);
template int lower_cost_desc<double>(const sgpmp_shape_t&, const sgpmp_cost_desc_t&, CostParams<double>&);

// Asynchronous global -> shared copies (SASS LDGSTS): the sample stream of K3 is staged through a per-THREAD ring.
template <int BYTES>
__device__ __forceinline__ void cp_async(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc), "n"(BYTES) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int PENDING>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(PENDING) : "memory"); }

// Ring depth (time steps in flight per thread) of cost_kernel's sample stream.  A thread walks T steps and needs the 2 n state
// components of step t before it can do anything with it; loaded just in time (round 1) every step began with a DRAM round trip
// (ncu, planar: 46 % of the stall samples on the first use of the loaded state, issue port 50 % busy, 0.34 of the HBM stream).
// With the ring the loads of step t + DEPTH - 1 are issued (LDGSTS, no destination registers) before step t is consumed, so
// DEPTH - 1 steps of HBM latency are covered per thread; every thread copies and reads ONLY ITS OWN slots (lane-consecutive
// words: conflict-free), so no barrier or mbarrier is involved — cp.async.wait_group orders a thread's own copies.  (A CTA-wide
// TMA ring with mbarriers was measured SLOWER than the just-in-time loads: profiles/r2/k3_tma_experiment.txt.)
template <int N> struct CostRing { static constexpr int DEPTH = N <= 4 ? 4 : (N <= 7 ? 3 : 2); };

template <typename real, int N, int CHAIN>
__global__ void __launch_bounds__(128)
cost_kernel(const __grid_constant__ CostParams<real> P, int G, int K, int S, int T,
            const double* __restrict__ tab, const real* __restrict__ samples, const real* __restrict__ means,
            real* __restrict__ costs, real* __restrict__ terms, size_t term_stride) {
    constexpr int d = 2 * N;
    constexpr int DP = (d + 3) & ~3;      // padded row length: rows stay 16-byte aligned for LDS.128
    constexpr int DEPTH = CostRing<N>::DEPTH;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    real* sph = reinterpret_cast<real*>(smem_raw);                       // [MAX_SPHERES][8] + coll_const
    real* bvec = sph + SPH_SMEM;                                         // [T][DP]
    double* tabDO = reinterpret_cast<double*>(bvec + (size_t)T * DP);    // [T][7]
    real* mu = reinterpret_cast<real*>(tabDO + (size_t)T * 7);           // [T][d]
    real* start = mu + (size_t)T * d;                                    // [d]
    real* goal = start + d;                                              // [d]
    real* ring = goal + d;                                               // [DEPTH][d][128]  per-thread slots

    const int NP = G * K;
    const int bp = blockIdx.x, b = bp / NP, p = bp - b * NP;
    if (means)
        for (int k = threadIdx.x; k < T * 7; k += blockDim.x)
            tabDO[k] = tab[(size_t)(k / 7) * SGPMP_TABLE_STRIDE + SGPMP_TAB_D11 + (k % 7)];
    if (means)
        for (int k = threadIdx.x; k < T * d; k += blockDim.x) mu[k] = means[(size_t)bp * T * d + k];
    stage_cta_constants<real, N, CHAIN>(P, b, p / K, G, start, goal, sph);
    double mub_part = 0.0;
    if (means) {
        for (int k = threadIdx.x; k < T * N; k += blockDim.x) {
            const int t = k / N, i = k - t * N;
            mub_part += precision_times_row<real>(tabDO, mu, T, N, t, i, &bvec[t * DP + i], &bvec[t * DP + N + i]);
        }
    }
    __shared__ double red64[32];
    const real mub = (real)block_sum_f64(mub_part, red64);

    const int s = blockIdx.y * blockDim.x + threadIdx.x;
    if (s >= S) return;
    CostSmem<real> sm;
    sm.start = start; sm.goal = goal; sm.bvec = means ? bvec : nullptr; sm.sph = sph;
    sm.coll_const = sph[SPH_STRIDE * SGPMP_MAX_SPHERES];
    sm.self_const = sph[SPH_STRIDE * SGPMP_MAX_SPHERES + 1];
    sm.mub = mub;
    sm.map = P.has_map ? P.occ_map + (size_t)(P.map_of_problem ? P.map_of_problem[b] : 0) * P.map_h * P.map_w : nullptr;
    sm.map_u8 = (P.has_map && P.occ_map_u8) ? P.occ_map_u8 + (size_t)(P.map_of_problem ? P.map_of_problem[b] : 0) * P.map_h * P.map_w : nullptr;

    TrajCost<real, N, CHAIN> tc;
    tc.begin();
    const real* xs = samples + (size_t)bp * T * d * S + s;
    real* my = ring + threadIdx.x;
    auto issue = [&](int t, int slot_w) {                 // step t into ring slot slot_w
        real* dst = my + (size_t)slot_w * d * 128;
        const real* src = xs + (size_t)t * d * S;
#pragma unroll
        for (int j = 0; j < d; ++j) cp_async<sizeof(real)>(dst + j * 128, src + (size_t)j * S);
    };
    auto consume = [&](int t, int slot_r) {               // step t out of ring slot slot_r = t % DEPTH
        cp_async_commit();                                // (an empty group near the end keeps the group count uniform)
        cp_async_wait<DEPTH - 1>();                       // the group of step t has landed
        const real* slot = my + (size_t)slot_r * d * 128;
        real x[d], y[d];
#pragma unroll
        for (int j = 0; j < d; ++j) {
            x[j] = slot[j * 128];
            y[j] = means ? x[j] - mu[t * d + j] : x[j];
        }
        tc.step(P, sm, t, T, x, y, y + N, means ? bvec + t * DP : nullptr);
    };
#pragma unroll
    for (int k = 0; k < DEPTH - 1; ++k) {
        if (k < T) issue(k, k);
        cp_async_commit();
    }
    if constexpr (CHAIN < 0) {
        // state-only body (short): the time loop is unrolled by the ring depth, so slot addresses are immediates
        for (int t0 = 0; t0 < T; t0 += DEPTH) {
#pragma unroll
            for (int k = 0; k < DEPTH; ++k) {
                const int t = t0 + k;
                if (t < T) {
                    if (t + DEPTH - 1 < T) issue(t + DEPTH - 1, (k + DEPTH - 1) % DEPTH);      // the slot step t - 1 was read from
                    consume(t, k);
                }
            }
        }
    } else {
        int wr = DEPTH - 1, rd = 0;                       // ring slots of the next step to load / to consume
        for (int t = 0; t < T; ++t) {
            if (t + DEPTH - 1 < T) { issue(t + DEPTH - 1, wr); wr = (wr + 1 == DEPTH) ? 0 : wr + 1; }
            consume(t, rd);
            rd = (rd + 1 == DEPTH) ? 0 : rd + 1;
        }
    }
    tc.finish(P, sm, T);
    const size_t o = (size_t)bp * S + s;
    costs[o] = tc.total();
    if (terms) {
        terms[SGPMP_TERM_START * term_stride + o] = tc.c_start;
        terms[SGPMP_TERM_GP * term_stride + o] = tc.c_gp;
        terms[SGPMP_TERM_GOAL * term_stride + o] = tc.c_goal;
        terms[SGPMP_TERM_COLL * term_stride + o] = tc.c_coll;
        terms[SGPMP_TERM_IS * term_stride + o] = tc.c_is;
        terms[SGPMP_TERM_SELF * term_stride + o] = tc.c_self;
        terms[SGPMP_TERM_EE * term_stride + o] = tc.c_ee;
    }
}

// Low-latency form of K3 for FEW trajectories (one planning problem): a trajectory's time steps are spread over the TW warps
// of a CTA (lane = sample, warp w takes t = w, w + TW, ...), so B*NP*S*TW threads work instead of B*NP*S — with one problem
// (2,048 samples) the thread-per-sample kernel leaves most of the GPU idle and every thread walks 64 dependent steps.
// Same per-step arithmetic (TrajCost::step on a fresh object with x_{t-1} preset); the per-step contributions are summed in a
// fixed order (warp 0..TW-1), so results are deterministic and agree with cost_kernel to fp32 rounding of the sum.
template <typename real, int N, int CHAIN, int TW, int SL>
__global__ void __launch_bounds__(32 * TW)
cost_st_kernel(const __grid_constant__ CostParams<real> P, int G, int K, int S, int T,
               const double* __restrict__ tab, const real* __restrict__ samples, const real* __restrict__ means,
               real* __restrict__ costs) {
    constexpr int d = 2 * N;
    constexpr int DP = (d + 3) & ~3;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    real* sph = reinterpret_cast<real*>(smem_raw);
    real* bvec = sph + SPH_SMEM;                                         // [T][DP]
    double* tabDO = reinterpret_cast<double*>(bvec + (size_t)T * DP);    // [T][7]
    real* mu = reinterpret_cast<real*>(tabDO + (size_t)T * 7);           // [T][d]
    real* start = mu + (size_t)T * d;
    real* goal = start + d;
    real* part = goal + d;                                               // [NSL][SL], NSL = 32 TW / SL time slices
    const int NP = G * K;
    const int bp = blockIdx.x, b = bp / NP, p = bp - b * NP;
    pdl_launch_dependents();
    for (int k = threadIdx.x; k < T * 7; k += blockDim.x)
        tabDO[k] = tab[(size_t)(k / 7) * SGPMP_TABLE_STRIDE + SGPMP_TAB_D11 + (k % 7)];
    stage_cta_constants<real, N, CHAIN>(P, b, p / K, G, start, goal, sph);
    pdl_wait();        // the tables and cost constants above are written by no kernel of the chain; means and samples are
    for (int k = threadIdx.x; k < T * d; k += blockDim.x) mu[k] = means[(size_t)bp * T * d + k];
    __syncthreads();
    double mub_part = 0.0;
    for (int k = threadIdx.x; k < T * N; k += blockDim.x) {
        const int t = k / N, i = k - t * N;
        mub_part += precision_times_row<real>(tabDO, mu, T, N, t, i, &bvec[t * DP + i], &bvec[t * DP + N + i]);
    }
    __shared__ double red64[32];
    const real mub = (real)block_sum_f64(mub_part, red64);
    CostSmem<real> sm;
    sm.start = start; sm.goal = goal; sm.bvec = bvec; sm.sph = sph;
    sm.coll_const = sph[SPH_STRIDE * SGPMP_MAX_SPHERES];
    sm.self_const = sph[SPH_STRIDE * SGPMP_MAX_SPHERES + 1];
    sm.mub = mub;
    sm.map = P.has_map ? P.occ_map + (size_t)(P.map_of_problem ? P.map_of_problem[b] : 0) * P.map_h * P.map_w : nullptr;
    sm.map_u8 = (P.has_map && P.occ_map_u8) ? P.occ_map_u8 + (size_t)(P.map_of_problem ? P.map_of_problem[b] : 0) * P.map_h * P.map_w : nullptr;

    // SL samples per CTA (consecutive threads = consecutive samples), 32 TW / SL time slices: slice w takes t = w, w + NSL, ...
    constexpr int NSL = 32 * TW / SL;
    const int lane = threadIdx.x % SL, w = threadIdx.x / SL;
    const int s = blockIdx.y * SL + lane;
    real acc = 0;
    if (s < S) {
        const real* xs = samples + (size_t)bp * T * d * S + s;
        for (int t = w; t < T; t += NSL) {
            TrajCost<real, N, CHAIN> tc;
            tc.begin();
            real x[d], y[d];
#pragma unroll
            for (int j = 0; j < d; ++j) {
                x[j] = xs[((size_t)t * d + j) * S];
                y[j] = x[j] - mu[t * d + j];
                tc.xp[j] = t > 0 ? xs[((size_t)(t - 1) * d + j) * S] : (real)0;
            }
            tc.step(P, sm, t, T, x, y, y + N, bvec + t * DP);
            real v = tc.partial(P, sm, T, t);
            if (CHAIN >= 0 && t == T - 1 && P.has_ee) {
                real q[N];
#pragma unroll
                for (int i = 0; i < N; ++i) q[i] = x[i];
                v += ee_se3_cost<real, N>(P, q) * P.ee_w;
            }
            acc += v;
        }
    }
    part[w * SL + lane] = acc;
    __syncthreads();
    if (w == 0 && s < S) {
        real tot = 0;
        for (int k = 0; k < NSL; ++k) tot += part[k * SL + lane];
        costs[(size_t)bp * S + s] = tot;
    }
}

template <typename real, int N, int CHAIN, int SL>
static int launch_cost_st_sl(const sgpmp_shape_t& sh, const CostParams<real>& P, const double* tables, const void* samples,
                             const void* means, void* costs, cudaStream_t st, bool pdl) {
    constexpr int TW = 16;                // 512 threads: SL samples x (512 / SL) time slices
    const int NP = sh.G * sh.K, d = 2 * N;
    dim3 grid((unsigned)(sh.B * NP), (unsigned)((sh.S + SL - 1) / SL));
    const size_t smem = (size_t)sh.T * 7 * sizeof(double) + ((size_t)sh.T * (d + ((d + 3) & ~3)) + 2 * d + SPH_SMEM + 32 * TW) * sizeof(real);
    if (smem > SGPMP_SMEM_OPTIN) {
        if (smem > 227 * 1024) { set_error("sgpmp_iterate_lowlat: T=%d too large for shared memory", sh.T); return SGPMP_ERR_UNSUPPORTED; }
        cudaFuncSetAttribute(cost_st_kernel<real, N, CHAIN, TW, SL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    launch_kernel(cost_st_kernel<real, N, CHAIN, TW, SL>, grid, dim3(32 * TW), smem, st, pdl, P, sh.G, sh.K, sh.S, sh.T, tables,
                  (const real*)samples, (const real*)means, (real*)costs);
    SGPMP_CHECK_LAUNCH("sgpmp_iterate_lowlat(cost)");
    return SGPMP_OK;
}

template <typename real, int N, int CHAIN>
static int launch_cost_st_n(const sgpmp_shape_t& sh, const CostParams<real>& P, const double* tables, const void* samples,
                            const void* means, void* costs, cudaStream_t st, bool pdl) {
    // 16 samples x 32 time slices per CTA while that still fits one wave of CTAs (one Panda problem: 128 CTAs, 12.8 us against
    // 17.2 us); 32 samples x 16 slices beyond (two problems: 37.9 against 41.6 us per iteration)
    const long ctas16 = (long)sh.B * sh.G * sh.K * ((sh.S + 15) / 16);
    if (ctas16 <= 148) return launch_cost_st_sl<real, N, CHAIN, 16>(sh, P, tables, samples, means, costs, st, pdl);
    return launch_cost_st_sl<real, N, CHAIN, 32>(sh, P, tables, samples, means, costs, st, pdl);
}

template <typename real>
static int launch_cost_st(const sgpmp_shape_t& sh, const sgpmp_cost_desc_t& desc, const double* tables, const void* samples,
                          const void* means, void* costs, cudaStream_t st, bool pdl) {
    CostParams<real> P;
    int rc = lower_cost_desc<real>(sh, desc, P);
    if (rc != SGPMP_OK) return rc;
    if constexpr (sizeof(real) == 4) {
        if (structured_fields_ok(P) && chain_is_panda_structure(desc, sh.n_dof))
            return P.has_self ? launch_cost_st_n<real, 7, 2>(sh, P, tables, samples, means, costs, st, pdl)
                              : launch_cost_st_n<real, 7, 1>(sh, P, tables, samples, means, costs, st, pdl);
    }
    const bool state_only = !P.has_spheres && !P.has_self && !P.has_ee;
    switch (sh.n_dof) {
#define SGPMP_DOF_CASE(N) case N: return state_only ? launch_cost_st_n<real, N, -1>(sh, P, tables, samples, means, costs, st, pdl) \
                                                    : launch_cost_st_n<real, N, 0>(sh, P, tables, samples, means, costs, st, pdl);
#include "sgpmp_dof_list.inc"
#undef SGPMP_DOF_CASE
        default:
            set_error("sgpmp_iterate_lowlat: n_dof=%d is not instantiated (see sgpmp_dof_list.inc)", sh.n_dof);
            return SGPMP_ERR_UNSUPPORTED;
    }
}

int cost_st_launch(const sgpmp_shape_t& sh, const sgpmp_cost_desc_t& desc, const double* tables, const void* samples,
                   const void* means, void* costs, cudaStream_t st, bool pdl) {
    if (sh.dtype == SGPMP_F32) return launch_cost_st<float>(sh, desc, tables, samples, means, costs, st, pdl);
    return launch_cost_st<double>(sh, desc, tables, samples, means, costs, st, pdl);
}

// Link-frame origins of N_cfg configurations: q [n_cfg][N] -> pos [n_cfg][L][3].  Same FK code as the cost
// kernel; used for known-answer tests and collision-freeness checks of final plans.
template <typename real, int N>
__global__ void fk_links_kernel(const __grid_constant__ CostParams<real> P, int n_cfg, const real* __restrict__ q,
                                real* __restrict__ pos) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cfg) return;
    real qq[N];
#pragma unroll
    for (int i = 0; i < N; ++i) qq[i] = q[(size_t)c * N + i];
    const int L = P.n_frames + (P.include_base ? 1 : 0);
    real* out = pos + (size_t)c * L * 3;
    int l = 0;
    fk_visit_links<real, N>(P, qq, [&](real x, real y, real z) {
        out[3 * l + 0] = x; out[3 * l + 1] = y; out[3 * l + 2] = z;
        ++l;
    });
}

template <typename real>
static int launch_fk(const sgpmp_cost_desc_t& desc, int n_dof, int n_cfg, const void* q, void* pos, cudaStream_t st) {
    sgpmp_shape_t sh;
    memset(&sh, 0, sizeof(sh));
    sh.n_dof = n_dof;
    CostParams<real> P;
    memset(&P, 0, sizeof(P));
    if (desc.n_frames < n_dof || desc.n_frames > SGPMP_MAX_FRAMES) { set_error("sgpmp_fk_link_positions: bad n_frames"); return SGPMP_ERR_INVALID_ARG; }
    for (int f = 0; f < desc.n_frames; ++f) {
        if (desc.chain_joint[f] != (f < n_dof ? f : -1)) { set_error("sgpmp_fk_link_positions: chain is not a serial arm"); return SGPMP_ERR_UNSUPPORTED; }
        for (int k = 0; k < 9; ++k) P.R[f][k] = (real)desc.chain_R[f][k];
        for (int k = 0; k < 3; ++k) P.p[f][k] = (real)desc.chain_p[f][k];
    }
    P.n_frames = desc.n_frames;
    P.include_base = desc.include_base;
    const int bs = 128;
    switch (n_dof) {
#define SGPMP_DOF_CASE(N) case N: fk_links_kernel<real, N><<<(n_cfg + bs - 1) / bs, bs, 0, st>>>(P, n_cfg, (const real*)q, (real*)pos); break;
#include "sgpmp_dof_list.inc"
#undef SGPMP_DOF_CASE
        default:
            set_error("sgpmp_fk_link_positions: n_dof=%d is not instantiated", n_dof);
            return SGPMP_ERR_UNSUPPORTED;
    }
    SGPMP_CHECK_LAUNCH("sgpmp_fk_link_positions");
    return SGPMP_OK;
}

template <typename real, int N, int CHAIN>
static int launch_cost_n(const sgpmp_shape_t& sh, const CostParams<real>& P, const double* tables, const void* samples,
                         const void* means, void* costs, void* terms, cudaStream_t st) {
    const int NP = sh.G * sh.K, d = 2 * N, bs = 128;
    dim3 grid((unsigned)(sh.B * NP), (unsigned)((sh.S + bs - 1) / bs));
    const size_t smem = (size_t)sh.T * 7 * sizeof(double) + ((size_t)sh.T * (d + ((d + 3) & ~3)) + 2 * d + SPH_SMEM +
                                                              (size_t)CostRing<N>::DEPTH * d * bs) * sizeof(real);
    if (smem > SGPMP_SMEM_OPTIN) {
        if (smem > 227 * 1024) { set_error("sgpmp_cost: T=%d too large for shared memory", sh.T); return SGPMP_ERR_UNSUPPORTED; }
        cudaFuncSetAttribute(cost_kernel<real, N, CHAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    cost_kernel<real, N, CHAIN><<<grid, bs, smem, st>>>(P, sh.G, sh.K, sh.S, sh.T, tables, (const real*)samples,
                                                  (const real*)means, (real*)costs, (real*)terms,
                                                  (size_t)sh.B * NP * sh.S);
    SGPMP_CHECK_LAUNCH("sgpmp_cost");
    return SGPMP_OK;
}

template <typename real>
static int launch_cost(const sgpmp_shape_t& sh, const sgpmp_cost_desc_t& desc, const double* tables, const void* samples,
                       const void* means, void* costs, void* terms, cudaStream_t st) {
    CostParams<real> P;
    int rc = lower_cost_desc<real>(sh, desc, P);
    if (rc != SGPMP_OK) return rc;
    if constexpr (sizeof(real) == 4) {
        if (structured_fields_ok(P) && chain_is_panda_structure(desc, sh.n_dof))
            return P.has_self ? launch_cost_n<real, 7, 2>(sh, P, tables, samples, means, costs, terms, st)
                              : launch_cost_n<real, 7, 1>(sh, P, tables, samples, means, costs, terms, st);
    }
    // no link fields and no EE goal: the instantiation without any FK / field code (the generic one carries ~4,000 instructions
    // of it, a stack frame and spills through the hot loop: planar K3 126 -> see profiles/r2 instructions per (sample, step))
    const bool state_only = !P.has_spheres && !P.has_self && !P.has_ee;
    switch (sh.n_dof) {
#define SGPMP_DOF_CASE(N) case N: return state_only ? launch_cost_n<real, N, -1>(sh, P, tables, samples, means, costs, terms, st) \
                                                    : launch_cost_n<real, N, 0>(sh, P, tables, samples, means, costs, terms, st);
#include "sgpmp_dof_list.inc"
#undef SGPMP_DOF_CASE
        default:
            set_error("sgpmp_cost: n_dof=%d is not instantiated (see sgpmp_dof_list.inc)", sh.n_dof);
            return SGPMP_ERR_UNSUPPORTED;
    }
}

}  // namespace sgpmp

using namespace sgpmp;

extern "C" int sgpmp_dof_supported(int32_t n_dof) {
    switch (n_dof) {
#define SGPMP_DOF_CASE(N) case N: return 1;
#include "sgpmp_dof_list.inc"
#undef SGPMP_DOF_CASE
        default: return 0;
    }
}

extern "C" int sgpmp_cost(const sgpmp_shape_t* shape, const sgpmp_cost_desc_t* desc, const double* tables,
                          const void* samples, const void* means, void* costs, void* terms, void* stream) {
    SGPMP_REQUIRE(shape_ok(shape), "sgpmp_cost: invalid shape");
    SGPMP_REQUIRE(desc && samples && costs, "sgpmp_cost: null pointer");
    SGPMP_REQUIRE(tables || !means, "sgpmp_cost: the IS term (means != NULL) needs the prior tables");
    if (shape->dtype == SGPMP_F32)
        return launch_cost<float>(*shape, *desc, tables, samples, means, costs, terms, (cudaStream_t)stream);
    return launch_cost<double>(*shape, *desc, tables, samples, means, costs, terms, (cudaStream_t)stream);
}

extern "C" int sgpmp_fk_link_positions(const sgpmp_cost_desc_t* desc, int32_t n_dof, int32_t dtype, int32_t n_cfg,
                                       const void* q, void* pos, void* stream) {
    SGPMP_REQUIRE(desc && q && pos && n_cfg > 0 && n_dof > 0, "sgpmp_fk_link_positions: bad arguments");
    SGPMP_REQUIRE(dtype == SGPMP_F32 || dtype == SGPMP_F64, "sgpmp_fk_link_positions: bad dtype");
    if (dtype == SGPMP_F32) return launch_fk<float>(*desc, n_dof, n_cfg, q, pos, (cudaStream_t)stream);
    return launch_fk<double>(*desc, n_dof, n_cfg, q, pos, (cudaStream_t)stream);
}
