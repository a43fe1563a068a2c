// Final plans: a collision check of every particle mean between and at its support states, and per problem the choice of the
// cheapest collision-free mean (sgpmp_select_plans).  No reference counterpart (DESIGN.md §7).
//
// States between support states are the constant-velocity GP prior's own interpolation (GPMP2's): per DoF,
//   x(tau) = Lambda(tau) x_i + Psi(tau) x_{i+1},   Psi = Q(tau) Phi(dt - tau)^T Q(dt)^-1,   Lambda = Phi(tau) - Psi Phi(dt),
// Phi(s) = [[1, s], [0, 1]], Q(s) = [[s^3/3, s^2/2], [s^2/2, s]] (Q_c cancels), which is cubic Hermite interpolation of (q, qdot).
// The kernels evaluate the same value as  Phi(tau) x_i + Psi (x_{i+1} - Phi(dt) x_i):  the entries of Lambda and Psi that act on
// q grow like 6/dt, and in fp32 their products with q cancel to the velocity with ~|q| 6/dt 2^-24 of error; the innovation
// x_{i+1} - Phi(dt) x_i is formed from differences of nearby values and keeps the interpolated state at fp32 resolution.
//
// Mapping: check kernel, one CTA of 128 threads per (problem, particle), thread per checked state; select kernel, one warp per
// problem.  The dense plan is written with the device function the check evaluates, so every dense state is a checked state.
#include <math.h>

#include "sgpmp_common.cuh"
#include "sgpmp_cost.cuh"

namespace sgpmp {

// Interpolation constants of one (dt, m): entry k - 1 belongs to tau_k = k dt / (m + 1), k = 1..m.  Host-computed in fp64.
template <typename real>
struct TimeInterp {
    real dt;
    real tau[SGPMP_MAX_TIME_INTERP];
    real psi[SGPMP_MAX_TIME_INTERP][4];   // Psi(tau_k), row-major
};

// State k of interval i: xa = x_i, xb = x_{i+1} (not read when k == 0: the support state itself, copied).
template <typename real, int N>
__device__ __forceinline__ void interp_state(const TimeInterp<real>& C, int k, const real* xa, const real* xb, real (&x)[2 * N]) {
    if (k == 0) {
#pragma unroll
        for (int j = 0; j < 2 * N; ++j) x[j] = xa[j];
        return;
    }
    const real tau = C.tau[k - 1], s0 = C.psi[k - 1][0], s1 = C.psi[k - 1][1], s2 = C.psi[k - 1][2], s3 = C.psi[k - 1][3];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        const real qa = xa[i], va = xa[N + i];
        const real ep = vfma(-C.dt, va, xb[i] - qa);          // x_{i+1} - Phi(dt) x_i
        const real ev = xb[N + i] - va;
        x[i] = vfma(s0, ep, vfma(s1, ev, vfma(tau, va, qa)));
        x[N + i] = vfma(s2, ep, vfma(s3, ev, va));
    }
}

template <typename real, int N>
__global__ void __launch_bounds__(128)
plan_check_kernel(const __grid_constant__ CostParams<real> P, const __grid_constant__ TimeInterp<real> C, int NP, int T, int m,
                  const real* __restrict__ means, real* __restrict__ clearance, int32_t* __restrict__ hits) {
    constexpr int d = 2 * N;
    __shared__ real sph[SGPMP_MAX_SPHERES * 4];
    __shared__ real md2[SGPMP_MAX_SPHERES][128];     // per thread and sphere: min |p - c|^2 over its points (sqrt is monotone, so
                                                     // one sqrt per sphere at the end gives min |p - c| - r exactly)
    __shared__ int red_h[4];
    const int bp = blockIdx.x, b = bp / NP;
    if (P.has_spheres) {
        for (int k = threadIdx.x; k < P.n_spheres * 4; k += 128)
            sph[k] = P.spheres[(size_t)(P.spheres_per_problem ? b : 0) * P.n_spheres * 4 + k];
        for (int o = 0; o < P.n_spheres; ++o) md2[o][threadIdx.x] = (real)INFINITY;
    }
    __syncthreads();
    const size_t map_off = P.has_map ? (size_t)(P.map_of_problem ? P.map_of_problem[b] : 0) * P.map_h * P.map_w : 0;
    const real* mu = means + (size_t)bp * T * d;
    const int n_points = (T - 1) * (m + 1) + 1;
    int nh = 0;
    // every state but t = 0: the planner cannot move the start state, and the collision cost skips it too
    for (int j = 1 + threadIdx.x; j < n_points; j += 128) {
        const int i = j / (m + 1), k = j - i * (m + 1);
        real x[d];
        interp_state<real, N>(C, k, mu + (size_t)i * d, mu + (size_t)(k ? i + 1 : i) * d, x);
        if (P.has_map) {
            const int c = map_cell(P, x[0], x[1]);
            nh += (P.occ_map_u8 ? P.occ_map_u8[map_off + c] != 0 : P.occ_map[map_off + c] != (real)0) ? 1 : 0;
        }
        if (P.has_spheres) {
            auto at = [&](real px, real py, real pz) {
#pragma unroll 1
                for (int o = 0; o < P.n_spheres; ++o) {
                    const real dx = px - sph[4 * o], dy = py - sph[4 * o + 1], dz = pz - sph[4 * o + 2];
                    md2[o][threadIdx.x] = vminv(md2[o][threadIdx.x], vfma(dx, dx, vfma(dy, dy, dz * dz)));
                }
            };
            // the sphere field's points: link-frame origins, then X_l + (X_{l+1} - X_l) alpha for l in [lo, hi)
            real PX[SGPMP_MAX_FRAMES + 1], PY[SGPMP_MAX_FRAMES + 1], PZ[SGPMP_MAX_FRAMES + 1];
            int L = 0;
            fk_visit_links<real, N>(P, x, [&](real px, real py, real pz) { PX[L] = px; PY[L] = py; PZ[L] = pz; ++L; });
#pragma unroll 1
            for (int l = 0; l < L; ++l) {
                at(PX[l], PY[l], PZ[l]);
                if (l >= P.sphere_interp_lo && l < P.sphere_interp_hi)
                    for (int a = 0; a < P.sphere_interp_n; ++a) {
                        const real al = P.sphere_alpha[a];
                        at(PX[l] + (PX[l + 1] - PX[l]) * al, PY[l] + (PY[l + 1] - PY[l]) * al, PZ[l] + (PZ[l + 1] - PZ[l]) * al);
                    }
            }
        }
    }
    // clearance = min_o (sqrt(min over the CTA's points of |p - c_o|^2) - r_o); hits: CTA sum
    __syncthreads();
    for (int h = 64; h > 0; h >>= 1) {
        if (threadIdx.x < h)
            for (int o = 0; o < P.n_spheres; ++o) md2[o][threadIdx.x] = vminv(md2[o][threadIdx.x], md2[o][threadIdx.x + h]);
        __syncthreads();
    }
    real best = (real)INFINITY;
    if (threadIdx.x < P.n_spheres) best = vsqrt(md2[threadIdx.x][0]) - sph[4 * threadIdx.x + 3];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        best = vminv(best, __shfl_xor_sync(0xffffffffu, best, o));
        nh += __shfl_xor_sync(0xffffffffu, nh, o);
    }
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) red_h[w] = nh;
    __syncthreads();
    if (threadIdx.x == 0) {
        nh = red_h[0] + red_h[1] + red_h[2] + red_h[3];
        clearance[bp] = best;
        hits[bp] = nh;
    }
}

// true if candidate (f1, c1, i1) ranks before (f2, c2, i2): feasible first, then lower cost (NaN last), then lower index
template <typename real>
__device__ __forceinline__ bool ranks_before(bool f1, real c1, int i1, bool f2, real c2, int i2) {
    if (f1 != f2) return f1;
    const bool n1 = isnan(c1), n2 = isnan(c2);
    if (n1 != n2) return n2;
    if (!n1 && c1 != c2) return c1 < c2;
    return i1 < i2;
}

template <typename real, int N>
__global__ void __launch_bounds__(128)
plan_select_kernel(const __grid_constant__ TimeInterp<real> C, int B, int NP, int T, int m, real margin,
                   const real* __restrict__ means, const real* __restrict__ costs, const real* __restrict__ clearance,
                   const int32_t* __restrict__ hits, int32_t* __restrict__ particle, int32_t* __restrict__ ok,
                   real* __restrict__ plan, real* __restrict__ dense) {
    constexpr int d = 2 * N;
    const int b = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (b >= B) return;
    bool bf = false;
    real bc = 0;
    int bi = NP;                  // NP: no candidate yet (every real index ranks before it)
    for (int p = lane; p < NP; p += 32) {
        const size_t o = (size_t)b * NP + p;
        const real c = costs[o];
        const bool f = hits[o] == 0 && clearance[o] >= margin && isfinite(c);
        if (bi == NP || ranks_before(f, c, p, bf, bc, bi)) { bf = f; bc = c; bi = p; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const bool f = __shfl_xor_sync(0xffffffffu, (int)bf, o) != 0;
        const real c = __shfl_xor_sync(0xffffffffu, bc, o);
        const int i = __shfl_xor_sync(0xffffffffu, bi, o);
        if (i != NP && (bi == NP || ranks_before(f, c, i, bf, bc, bi))) { bf = f; bc = c; bi = i; }
    }
    if (lane == 0) { particle[b] = bi; ok[b] = bf ? 1 : 0; }
    const real* mu = means + ((size_t)b * NP + bi) * T * d;
    for (int k = lane; k < T * d; k += 32) plan[(size_t)b * T * d + k] = mu[k];
    if (dense) {
        const int n_points = (T - 1) * (m + 1) + 1;
        real* out = dense + (size_t)b * n_points * d;
        for (int j = lane; j < n_points; j += 32) {
            const int i = j / (m + 1), k = j - i * (m + 1);
            real x[d];
            interp_state<real, N>(C, k, mu + (size_t)i * d, mu + (size_t)(k ? i + 1 : i) * d, x);
#pragma unroll
            for (int q = 0; q < d; ++q) out[(size_t)j * d + q] = x[q];
        }
    }
}

template <typename real>
static int launch_select_plans(const sgpmp_shape_t& sh, const sgpmp_cost_desc_t& desc, int m, double margin, const void* means,
                               const void* costs, void* clearance, int32_t* hits, int32_t* particle, int32_t* ok, void* plan,
                               void* dense, cudaStream_t st) {
    CostParams<real> P;
    int rc = lower_cost_desc<real>(sh, desc, P);
    if (rc != SGPMP_OK) return rc;
    TimeInterp<real> C;
    memset(&C, 0, sizeof(C));
    const double dt = desc.dt;
    C.dt = (real)dt;
    // Q(dt)^-1 = (12 / dt^4) [[dt, -dt^2/2], [-dt^2/2, dt^3/3]]
    const double w = 12.0 / (dt * dt * dt * dt);
    const double qi00 = w * dt, qi01 = -w * dt * dt / 2, qi11 = w * dt * dt * dt / 3;
    for (int k = 1; k <= m; ++k) {
        const double tau = k * dt / (m + 1), u = dt - tau;
        // A = Q(tau) Phi(dt - tau)^T,  Phi(u)^T = [[1, 0], [u, 1]]
        const double a00 = tau * tau * tau / 3 + u * tau * tau / 2, a01 = tau * tau / 2;
        const double a10 = tau * tau / 2 + u * tau, a11 = tau;
        C.tau[k - 1] = (real)tau;
        C.psi[k - 1][0] = (real)(a00 * qi00 + a01 * qi01);
        C.psi[k - 1][1] = (real)(a00 * qi01 + a01 * qi11);
        C.psi[k - 1][2] = (real)(a10 * qi00 + a11 * qi01);
        C.psi[k - 1][3] = (real)(a10 * qi01 + a11 * qi11);
    }
    const int NP = sh.G * sh.K;
    switch (sh.n_dof) {
#define SGPMP_DOF_CASE(N)                                                                                                        \
    case N:                                                                                                                      \
        plan_check_kernel<real, N><<<(unsigned)(sh.B * NP), 128, 0, st>>>(P, C, NP, sh.T, m, (const real*)means,               \
                                                                         (real*)clearance, hits);                               \
        SGPMP_CHECK_LAUNCH("sgpmp_select_plans(check)");                                                                         \
        plan_select_kernel<real, N><<<(unsigned)((sh.B + 3) / 4), 128, 0, st>>>(C, sh.B, NP, sh.T, m, (real)margin,             \
                                                                               (const real*)means, (const real*)costs,          \
                                                                               (const real*)clearance, hits, particle, ok,      \
                                                                               (real*)plan, (real*)dense);                      \
        SGPMP_CHECK_LAUNCH("sgpmp_select_plans(select)");                                                                        \
        return SGPMP_OK;
#include "sgpmp_dof_list.inc"
#undef SGPMP_DOF_CASE
        default:
            set_error("sgpmp_select_plans: n_dof=%d is not instantiated (see sgpmp_dof_list.inc)", sh.n_dof);
            return SGPMP_ERR_UNSUPPORTED;
    }
}

}  // namespace sgpmp

using namespace sgpmp;

extern "C" int sgpmp_select_plans(const sgpmp_shape_t* shape, const sgpmp_cost_desc_t* desc, int32_t n_interp, double margin,
                                  const void* means, const void* costs, void* clearance, int32_t* hits, int32_t* particle,
                                  int32_t* ok, void* plan, void* dense, void* stream) {
    SGPMP_REQUIRE(shape_ok(shape), "sgpmp_select_plans: invalid shape");
    SGPMP_REQUIRE(desc && means && costs && clearance && hits && particle && ok && plan, "sgpmp_select_plans: null pointer");
    SGPMP_REQUIRE(n_interp >= 0 && n_interp <= SGPMP_MAX_TIME_INTERP, "sgpmp_select_plans: n_interp=%d is outside [0, %d]", n_interp,
                  SGPMP_MAX_TIME_INTERP);
    SGPMP_REQUIRE(isfinite(margin), "sgpmp_select_plans: margin must be finite, got %g", margin);
    if (shape->dtype == SGPMP_F32)
        return launch_select_plans<float>(*shape, *desc, n_interp, margin, means, costs, clearance, hits, particle, ok, plan, dense,
                                          (cudaStream_t)stream);
    return launch_select_plans<double>(*shape, *desc, n_interp, margin, means, costs, clearance, hits, particle, ok, plan, dense,
                                       (cudaStream_t)stream);
}
