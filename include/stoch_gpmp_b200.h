/*
 * stoch_gpmp_b200 — C-ABI of the B200-native StochGPMP hot path.
 *
 * This header is the drop-in boundary: plain pointers and sizes, no torch types.  Every entry point
 * replaces one piece of arithmetic that the reference (anindex/stoch_gpmp, pure Python on PyTorch)
 * performs inside `StochGPMP.reset()/optimize()`; the citation on each function is the reference
 * file:line it stands in for.  The reference-side binding (ctypes) is shown in INTEGRATION.md and
 * implemented in stoch_gpmp_b200/_lib.py.
 *
 * Conventions
 *   - all array arguments are DEVICE pointers unless marked (host);
 *   - `dtype` selects the arithmetic/storage type `real` of every `void*` array: SGPMP_F32 or SGPMP_F64;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); calls are asynchronous,
 *     nothing here synchronises the device;
 *   - every function returns an sgpmp status code (0 = OK) and never throws; sgpmp_last_error()
 *     gives a thread-local text for the last non-OK status;
 *   - shapes: B problems, G goals, K particle means per goal, NP = G*K particles, S samples per
 *     particle, T support states, n DoF, d = 2n (state = [pos(n), vel(n)]), M = T*d.
 *
 * Memory layouts (row-major, last index fastest)
 *   means    [B, NP, T, d]      == reference `particle_means` [NP,T,d] per problem (planner.py:215)
 *   samples  [B, NP, T, d, S]   "S-minor": consecutive samples are consecutive in memory so that one
 *                               thread per sample reads/writes fully coalesced.  The reference's logical
 *                               `state_samples[p, s, t, j]` (planner.py:243, itself a non-contiguous
 *                               transposed view) is samples[b, p, t, j, s]; the Python host returns
 *                               permuted views, no copy.
 *   eps      same layout as samples
 *   costs / weights [B, NP, S]
 *   tables   [T, SGPMP_TABLE_STRIDE] doubles per prior, see sgpmp_prior_factor
 */
#ifndef STOCH_GPMP_B200_H
#define STOCH_GPMP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SGPMP_ABI_VERSION 7

enum { SGPMP_F32 = 0, SGPMP_F64 = 1 };

enum {
    SGPMP_OK = 0,
    SGPMP_ERR_INVALID_ARG = 1,
    SGPMP_ERR_UNSUPPORTED = 2, /* shape not instantiated (e.g. n_dof) — the host raises NotImplementedError */
    SGPMP_ERR_CUDA = 3,
    SGPMP_ERR_NO_DEVICE = 4
};

#define SGPMP_TABLE_STRIDE 16
/* column indices of one table row (time step t, one DoF; all DoF share the tables) */
enum {
    SGPMP_TAB_G11 = 0, SGPMP_TAB_G21 = 1, SGPMP_TAB_G22 = 2,                      /* G_t = A_t^-T (lower)          */
    SGPMP_TAB_H11 = 3, SGPMP_TAB_H12 = 4, SGPMP_TAB_H21 = 5, SGPMP_TAB_H22 = 6,   /* H_t = G_t C_{t-1}^T, H_0 = 0  */
    SGPMP_TAB_D11 = 7, SGPMP_TAB_D12 = 8, SGPMP_TAB_D22 = 9,                      /* P[t,t]                        */
    SGPMP_TAB_O11 = 10, SGPMP_TAB_O12 = 11, SGPMP_TAB_O21 = 12, SGPMP_TAB_O22 = 13 /* P[t+1,t] (zero row T-1)      */
};

#define SGPMP_MAX_FRAMES 16
#define SGPMP_MAX_SPHERES 16
#define SGPMP_MAX_INTERP 8        /* link interpolation: extra points per link pair */
#define SGPMP_MAX_LINK_POINTS 48  /* link frames + interpolated points of one field */
#define SGPMP_MAX_TIME_INTERP 32  /* sgpmp_select_plans: states checked between two support states */
#define SGPMP_NUM_TERMS 7
/* total = (((((start + gp) + goal) + self) + coll) + ee) + is  — the order of the shipped cost lists
 * (examples/panda_environment.py:90), then the IS term (planner.py:236) */
enum { SGPMP_TERM_START = 0, SGPMP_TERM_GP = 1, SGPMP_TERM_GOAL = 2, SGPMP_TERM_COLL = 3, SGPMP_TERM_IS = 4, SGPMP_TERM_SELF = 5,
       SGPMP_TERM_EE = 6 };

/* Problem-batch shape.  problem_gid0 is the GLOBAL index of problem 0 of this shard: the Philox
 * counters are keyed by global problem/particle ids so that results do not depend on how the batch is
 * sharded over GPUs; sample_gid0 does the same for a particle's samples in split-particle mode. */
typedef struct sgpmp_shape {
    int32_t B, G, K, S, T, n_dof;
    int32_t dtype;
    int32_t sample_gid0;   /* global index of sample 0 of this rank's slice (split-particle mode), else 0 */
    int64_t problem_gid0;
} sgpmp_shape_t;

/* Lowered form of the reference's cost objects (what StochGPMP.__init__ extracts from cost.cost_list):
 *   CostGP          cost_functions.py:90-146   sigma_start, sigma_gp, start_state, dt   (CostGPTrajectory :171-218: no start factor)
 *   CostGoalPrior   cost_functions.py:342-388  sigma_goal_prior, multi_goal_states
 *   CostCollision   cost_functions.py:223-261  sigma_coll + field:
 *       ObstacleMap         envs/obst_map.py:108-188     (occupancy grid lookup)
 *       LinkDistanceField   costs/fields.py:30-86 'rbf'  (FK link positions vs obstacle spheres)
 *       LinkSelfDistanceField costs/fields.py:89-127     (FK link positions vs each other; own sigma)
 *   CostGoal        cost_functions.py:282-321  sigma_goal + EESE3DistanceField (costs/fields.py:130-153): SE(3) distance
 *                                              of the LAST link frame to a target pose at the LAST time step
 *   IS term         planner.py:233-236         temperature * x^T Sigma^-1 mu
 * FK chain = the callable the reference passes as CostComposite(FK=...) (cost_functions.py:39-52),
 * restated as a serial chain of fixed transforms + revolute z joints. */
typedef struct sgpmp_cost_desc {
    double dt;
    double sigma_start;       /* <= 0: no start factor (CostGPTrajectory, cost_functions.py:171-218) */
    double sigma_gp;
    double sigma_goal_prior;  /* <= 0: no CostGoalPrior term */
    double temperature;       /* weight of the IS term; 0 disables it */

    const void* start;        /* [B, d] real */
    const void* goals;        /* [B, G, d] real, or NULL */

    /* occupancy map field (NULL = absent) */
    const void* occ_map;             /* [n_maps, map_h, map_w] real; value = map[iy][ix] */
    const int32_t* map_of_problem;   /* [B] map index per problem, or NULL => map 0 */
    int32_t n_maps, map_h, map_w;
    int32_t origin_xi, origin_yi;
    int32_t reserved0;
    double map_inv_cell;             /* 1/cell_size exactly as the reference forms it (obst_map.py:172) */
    double map_sigma_coll;

    /* sphere field (NULL = absent); needs the FK chain */
    const void* spheres;             /* [B, n_spheres, 4] or [n_spheres, 4] real: (cx, cy, cz, r) */
    int32_t n_spheres;
    int32_t spheres_per_problem;     /* 1: [B,O,4]; 0: one set shared by all problems */
    double sphere_sigma_coll;

    /* FK chain (host data, copied into kernel parameters) */
    int32_t n_frames;                /* <= SGPMP_MAX_FRAMES; frames after the base */
    int32_t include_base;            /* 1: the base frame (identity, origin) is also a link position */
    double chain_R[SGPMP_MAX_FRAMES][9];  /* fixed rotation parent->child, row-major */
    double chain_p[SGPMP_MAX_FRAMES][3];  /* fixed translation parent->child */
    int32_t chain_joint[SGPMP_MAX_FRAMES];/* joint index rotating about child z, or -1 (fixed) */

    /* self-collision field (needs the FK chain): sum_{i,j} exp(-|p_i - p_j|^2 / (2 margin^2)) over all ordered
     * pairs of link frames incl. i == j, weight 1/self_sigma_coll^2 */
    double self_margin;              /* <= 0: absent */
    double self_sigma_coll;

    /* optional byte copy of occ_map ([n_maps, map_h, map_w] uint8, same values: occupancy COUNTS are small
     * integers, envs/obst_map.py:71,104).  When non-NULL the kernels gather from it instead of occ_map: a 200x200
     * map is 40 KB instead of 160 KB (fp32), so it stays L1-resident.  Bit-exact: every count <= 255 is exact in fp32/fp64. */
    const uint8_t* occ_map_u8;

    /* LinkDistanceField.field_type (costs/fields.py:78-86): how the sphere field combines link origins p and spheres (c, r)
     *   SGPMP_FIELD_RBF        sum exp(-0.5 |p - c|^2 / r^2)
     *   SGPMP_FIELD_SDF        max (r - |p - c|);  SGPMP_FIELD_SDF_CLAMPED: max min(r - |p - c|, 0)   (clamp_sdf=True)
     *   SGPMP_FIELD_OCCUPANCY  number of (link, sphere) pairs with |p - c| < r */
    int32_t sphere_field_type;
    int32_t reserved1;

    /* Link interpolation (LinkDistanceField / LinkSelfDistanceField num_interpolate, link_interpolate_range;
     * costs/fields.py:68-74, :117-123): for i in [lo, hi) the points X_i + (X_{i+1} - X_i) alpha_k, k < n, are appended to the
     * link-frame origins (indices count the base frame when include_base).  alpha is host data: the reference evaluates
     * torch.linspace(0, 1, n + 2)[1:n+1] in float32 and casts it, so the host passes exactly those values.  n = 0: off. */
    int32_t sphere_interp_n, sphere_interp_lo, sphere_interp_hi;
    int32_t self_interp_n, self_interp_lo, self_interp_hi;
    double sphere_interp_alpha[SGPMP_MAX_INTERP];
    double self_interp_alpha[SGPMP_MAX_INTERP];

    /* End-effector SE(3) goal (CostGoal + EESE3DistanceField; needs the FK chain):
     *   dist = ee_w_pos |p_ee - p*| + ee_w_rot acos(clamp((tr(R_ee^T R*) - 1)/2, -1, 1)),  cost = dist^2 (ee_square) or dist,
     *   weight 1/ee_sigma_goal^2, evaluated on the last link frame at t = T-1 only.
     * SE3_distance itself lives in the absent torch_robotics: this definition is oracle/se3.py's (parity unpinned there). */
    double ee_sigma_goal;            /* <= 0: absent */
    double ee_target_R[9];           /* target rotation, row-major */
    double ee_target_p[3];
    double ee_w_pos, ee_w_rot;
    int32_t ee_square;
    int32_t reserved2;
} sgpmp_cost_desc_t;

enum { SGPMP_FIELD_RBF = 0, SGPMP_FIELD_SDF = 1, SGPMP_FIELD_SDF_CLAMPED = 2, SGPMP_FIELD_OCCUPANCY = 3 };

int sgpmp_abi_version(void);
const char* sgpmp_last_error(void);
/* 1 if the cost / fused kernels are instantiated for this DoF count (sampling / prior are generic). */
int sgpmp_dof_supported(int32_t n_dof);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches counter) */
int64_t sgpmp_launch_count(void);

/* K1 — prior factor.  Replaces MultivariateNormal(precision_matrix=...) construction
 * (mp_priors_multi.py:100-110 -> torch multivariate_normal.py:79-85) for the block-tridiagonal
 * constant-velocity precision of mp_priors_multi.py:170-202, per DoF (2x2 blocks), in fp64.
 *   D [n_priors, T, 3]   (d11, d12, d22) of P[t,t]
 *   O [n_priors, T-1, 4] (o11, o12, o21, o22) of P[t+1,t]
 *   tables [n_priors, T, 16] out;  not_pd [n_priors] out: 0, or 1 + index of the failing pivot block
 * One thread per prior runs the reverse block Cholesky P = U U^T. */
int sgpmp_prior_factor(int32_t n_priors, int32_t T, const double* D, const double* O,
                       double* tables, int32_t* not_pd, void* stream);

/* Dense scale_tril L [M, M] (row-major, `dtype`) expanded from one prior's tables — the matrix the
 * reference holds as dist._unbroadcasted_scale_tril (multivariate_normal.py:196).  Test / interop aid. */
int sgpmp_prior_dense_L(int32_t T, int32_t n_dof, const double* tables, int32_t dtype, void* L, void* stream);

/* K2 — sampling x = mu + L eps (mp_priors_multi.py:204-207 -> multivariate_normal.py:251-254) as the
 * banded recurrence y_t = G_t eps_t - H_t y_{t-1}.
 *   eps_in  NULL: draw eps in-kernel (Philox4x32-10 keyed by seed/draw/global ids);
 *           else: use these normals (parity with the reference's torch-drawn eps)
 *   eps_out optional: the normals that were used
 * Here the "particles" axis is generic: for the INIT prior pass G as NP (K=1 in shape) and S = K. */
int sgpmp_sample(const sgpmp_shape_t* shape, const double* tables, const void* means,
                 const void* eps_in, uint64_t seed, uint32_t draw,
                 void* samples, void* eps_out, void* stream);

/* K3 — per-trajectory-sample cost: CostComposite.eval (cost_functions.py:47-58) + the IS term
 * (planner.py:229-237).  costs [B,NP,S]; terms optional [SGPMP_NUM_TERMS, B, NP, S] (SGPMP_TERM_* order).
 * means == NULL drops the IS term (then tables may be NULL): that is CostComposite.eval alone. */
int sgpmp_cost(const sgpmp_shape_t* shape, const sgpmp_cost_desc_t* desc, const double* tables,
               const void* samples, const void* means, void* costs, void* terms, void* stream);

/* Link-frame origins by the same FK code the cost kernel uses: q [n_cfg, n_dof] -> pos [n_cfg, L, 3],
 * L = n_frames + include_base; only the chain fields of `desc` are read.  Stands in for the FK callable
 * of CostComposite (cost_functions.py:51-52) when checking collision-freeness of final plans. */
int sgpmp_fk_link_positions(const sgpmp_cost_desc_t* desc, int32_t n_dof, int32_t dtype, int32_t n_cfg,
                            const void* q, void* pos, void* stream);

/* Final plans (no reference counterpart; the reference's _get_traj('best') takes one argmax over the weights of all samples):
 * a collision check of every particle mean and, per problem, the best collision-free one.  Two launches, no synchronisation.
 *   means      [B,NP,T,d]; costs [B,NP] the ranking cost of each mean (sgpmp_cost with S = 1 and means == NULL)
 *   n_interp   m in [0, SGPMP_MAX_TIME_INTERP]: every mean is checked at P = (T-1)(m+1)+1 states; point j lies in interval
 *              i = j/(m+1) at tau = (j%(m+1)) dt/(m+1) and is the constant-velocity GP prior's interpolation
 *              x(tau) = Lambda(tau) x_i + Psi(tau) x_{i+1} per DoF (cubic Hermite in (q, qdot)); tau = 0 is x_i itself
 *   clearance  [B,NP] out: min over the checked states (all but t = 0) of |p - c| - r over the sphere field's points (link-frame
 *              origins + its link interpolation) and spheres; +inf without a sphere field.  The self-collision field is not checked.
 *   hits       [B,NP] out: number of checked states whose occupancy-map cell is non-zero; 0 without a map
 *   particle   [B] out: argmin cost over the feasible particles (hits == 0, clearance >= margin, finite cost), ties to the lowest
 *              index; with none feasible the argmin over all (NaN last) and ok = 0.   ok [B] out: 1 if the chosen one is feasible
 *   plan       [B,T,d] out: means[b, particle[b]] bit for bit;  dense [B,P,d] out (may be NULL): its checked states */
int sgpmp_select_plans(const sgpmp_shape_t* shape, const sgpmp_cost_desc_t* desc, int32_t n_interp, double margin,
                       const void* means, const void* costs, void* clearance, int32_t* hits, int32_t* particle, int32_t* ok,
                       void* plan, void* dense, void* stream);

/* K4 — softmax over the S samples of each particle + weighted-mean update
 * (StochGPMP._update_distribution, planner.py:263-275).  means is updated in place;
 * grad [B,NP,T,d] and weights [B,NP,S] are optional outputs. */
int sgpmp_update(const sgpmp_shape_t* shape, double temperature, double step_size,
                 const void* costs, const void* samples, void* means, void* grad, void* weights,
                 void* stream);

/* Fused optimisation loop: n_iters iterations of sample -> cost -> softmax -> update
 * (StochGPMP.optimize, planner.py:277-317) in ONE launch, one CTA per (problem, particle); samples are
 * never written to HBM except, optionally, those of the last iteration.
 *   eps_in     NULL (in-kernel Philox, draw index = draw0 + iteration) or [n_iters, B, NP, T, d, S]
 *   means      in/out; means_pre out (optional): the means BEFORE the last iteration's update, which is
 *              what optimize() returns (planner.py:252-253)
 *   samples    optional out, last iteration only;  costs/weights/grad optional outs, last iteration */
int sgpmp_iterate(const sgpmp_shape_t* shape, const sgpmp_cost_desc_t* desc, const double* tables,
                  double step_size, int32_t n_iters, const void* eps_in, uint64_t seed, uint32_t draw0,
                  void* means, void* means_pre, void* samples, void* costs, void* weights, void* grad,
                  void* stream);

/* The same loop for FEW problems (the reference's own use: one problem per planner), where the fused kernel's thread-per-sample
 * mapping leaves the GPU idle: per iteration three short launches — sgpmp_sample (thread per sample and DoF), a cost kernel with
 * thread per (sample, time slice), sgpmp_update with the state rows of a particle divided over CTAs — all n_iters iterations
 * enqueued by this one call.  Same arguments and results as sgpmp_iterate (same Philox stream; costs agree to the fp rounding
 * of the per-step sum), except that the sample workspace [B,NP,T,d,S] and costs [B,NP,S] are REQUIRED: samples_ws holds the
 * last iteration's samples on return. */
int sgpmp_iterate_lowlat(const sgpmp_shape_t* shape, const sgpmp_cost_desc_t* desc, const double* tables,
                         double step_size, int32_t n_iters, const void* eps_in, uint64_t seed, uint32_t draw0,
                         void* means, void* means_pre, void* samples_ws, void* costs, void* weights, void* grad,
                         void* stream);

/* Split-particle mode (one problem's samples sharded over ranks, SURVEY §8e).  Local statistics of
 * this rank's S_local samples per particle:  stats[B,NP, 2 + M] = (m, Z, A[M]) with
 *   m = max_s(-c_s/tau), Z = sum_s exp(-c_s/tau - m), A = sum_s exp(-c_s/tau - m) eps_s.
 * After the cross-rank log-sum-exp merge (NCCL, done by the host), sgpmp_apply_stats applies
 * mu += step * L (A/Z). */
int sgpmp_local_stats(const sgpmp_shape_t* shape, double temperature, const void* costs, const void* eps,
                      void* stats, void* stream);
int sgpmp_apply_stats(const sgpmp_shape_t* shape, const double* tables, double step_size,
                      const void* stats, void* means, void* grad, void* stream);

/* Split-particle mode without materialised samples (round 2).  The arithmetic being split is the reference's
 * _update_distribution, stoch_gpmp/planner.py:263-275 (softmax over ALL S samples of a particle, weighted mean update).
 *
 * sgpmp_iterate_stats: ONE fused launch over the samples [shape->sample_gid0, + shape->S) of every particle: sample -> cost
 *   -> local softmax statistics  stats[B,NP, 2 + M] = (m, Z, A)  (definitions above); `means` are read only, `costs`
 *   [B,NP,S] is optional.  The weighted eps-sum is regenerated from the counter-based RNG stream, nothing is materialised.
 * sgpmp_merge_apply_stats: stats_all [n_ranks][B,NP, 2 + M] are merged by log-sum-exp in rank order inside the kernel
 *   (m = max_r m_r, Z = sum_r Z_r e^(m_r - m), A = sum_r A_r e^(m_r - m)) and mu += step L (A/Z) is applied; grad optional.
 * sgpmp_comm_*: an NCCL communicator owned by this library (libnccl is resolved with dlopen at run time; sgpmp_nccl_load
 *   may name its path first).  Rank 0 calls sgpmp_comm_unique_id, the 128 bytes travel to the other ranks by any means
 *   (the Python host uses torch.distributed), every rank calls sgpmp_comm_init.
 * sgpmp_allreduce_stats: the exchange step — ncclAllGather of the local blocks into stats_all on `stream` (SURVEY 8b).
 * sgpmp_iterate_split_particles: n_iters iterations of  iterate_stats -> all_gather -> merge_apply  enqueued on `stream`
 *   by one call (no host synchronisation; comm may be NULL iff n_ranks == 1).  means_pre (optional) receives the means
 *   before the LAST update, costs (optional) this rank's costs and grad (optional) the gradient of the last iteration. */
int sgpmp_iterate_stats(const sgpmp_shape_t* shape, const sgpmp_cost_desc_t* desc, const double* tables,
                        uint64_t seed, uint32_t draw, const void* means, void* costs, void* stats, void* stream);
int sgpmp_merge_apply_stats(const sgpmp_shape_t* shape, const double* tables, double step_size, const void* stats_all,
                            int32_t n_ranks, void* means, void* grad, void* stream);
int sgpmp_nccl_load(const char* path);
int sgpmp_comm_unique_id(void* id128);
int sgpmp_comm_init(const void* id128, int32_t rank, int32_t n_ranks, void** comm);
int sgpmp_comm_destroy(void* comm);
int sgpmp_allreduce_stats(void* comm, const sgpmp_shape_t* shape, const void* stats_local, void* stats_all, void* stream);
int sgpmp_iterate_split_particles(const sgpmp_shape_t* shape_local, const sgpmp_cost_desc_t* desc, const double* tables,
                                  double step_size, int32_t n_iters, uint64_t seed, uint32_t draw0, void* means,
                                  void* means_pre, void* comm, int32_t n_ranks, void* stats_local, void* stats_all,
                                  void* costs, void* grad, void* stream);

/* Gauss-Newton GPMP (the reference's second planner, stoch_gpmp/planner.py:352-661; SURVEY §8f rank 4): n_iters iterations of
 *   A, b, K = cost.get_linear_system(means)  (cost_functions.py:60-85);  J^T J = A^T K A + damping  (planner.py:602-617);
 *   d_theta = solve(J^T J, A^T K b)  (planner.py:619-633);  means += step_size d_theta  (planner.py:592)
 * on the block-tridiagonal structure of J^T J (never formed densely), two launches per iteration, fp64 arithmetic.
 *   shape      B, G, K, T, n_dof, dtype (S is ignored: GPMP draws no samples)
 *   desc       CostGP + CostGoalPrior + link fields ('rbf' sphere field, self-collision field; with interpolation) + the EE
 *              SE(3) goal.  The occupancy map (a floor() lookup: no gradient) and the sdf / occupancy sphere fields are
 *              SGPMP_ERR_UNSUPPORTED here.
 *   D, O       [T,3] / [T-1,4] per-DoF 2x2 blocks of the start/GP/goal part of A^T K A — the closed form of
 *              sgpmp_prior_factor's inputs evaluated with the COST sigmas (sigma_start, sigma_gp, sigma_goal_prior)
 *   delta, trust_region   damping: delta I, or delta diag(mean over the particles of a problem of A^T K A)
 *   method     SGPMP_GPMP_INVERSE: d = (J^T J)^-1 g.  SGPMP_GPMP_CHOLESKY: the reference's branch AS WRITTEN
 *              (planner.py:626-629 passes l^T with upper=False to the second triangular solve): d = diag(l)^-1 l^-1 g
 *   means      in/out [B,NP,T,d];  d_theta optional out (last iteration);  costs out [B,NP] = b^T K b of the LAST
 *              linear system, i.e. at the means before the last update (planner.py:545,635-637)
 *   not_pd     out [B*NP] int32: 0, or 1 + index of the first pivot block that is not positive definite
 *   workspace  device scratch of sgpmp_gpmp_workspace_bytes(shape, method) bytes */
enum { SGPMP_GPMP_INVERSE = 0, SGPMP_GPMP_CHOLESKY = 1 };
int64_t sgpmp_gpmp_workspace_bytes(const sgpmp_shape_t* shape, int32_t method);
int sgpmp_gpmp_step(const sgpmp_shape_t* shape, const sgpmp_cost_desc_t* desc, const double* D, const double* O,
                    double delta, int32_t trust_region, int32_t method, double step_size, int32_t n_iters,
                    void* means, void* d_theta, void* costs, void* workspace, int64_t workspace_bytes,
                    int32_t* not_pd, void* stream);

/* K2, dense-L variant on the tensor cores (the reference's formulation: loc + L @ eps, multivariate_normal.py:251-254, per DoF
 * because the precision decouples; SURVEY §8(d) "second K2 variant"): samples = means + L1 eps_in with L1 [2T, 2T] the per-DoF
 * scale_tril (sgpmp_prior_dense_L with n_dof = 1), tcgen05 kind::tf32 with a 3xTF32 split.  fp32 only; eps_in is required.
 * Not the product path (32x the flops of the banded recurrence) — a measured comparison point, see bench_kernels.py. */
int sgpmp_sample_dense_tc(const sgpmp_shape_t* shape, const void* L1, const void* means, const void* eps_in,
                          void* samples, void* stream);

/* Weighted sample covariance of every particle (diagnostic; NO reference counterpart — the reference keeps Sigma^-1 fixed,
 * planner.py:226; asked for by the north-star next to the weighted-mean update of planner.py:263-275):
 *   cov[b,p] = sum_s w[b,p,s] (x_s - mu)(x_s - mu)^T      samples [B,NP,T,d,S] (S-minor), means [B,NP,T,d], weights [B,NP,S]
 *   cov out  [B,NP,M,M], M = T*d.
 * fp32 with use_tensor_cores != 0: tcgen05.mma kind::tf32 with a 3xTF32 split (accumulator in TMEM); otherwise (and always
 * for fp64) a CUDA-core kernel with fp64 accumulation.  B*NP <= 65535. */
int sgpmp_weighted_cov(const sgpmp_shape_t* shape, const void* samples, const void* means, const void* weights,
                       void* cov, int32_t use_tensor_cores, void* stream);

/* Pipe-peak probes for the roofline denominators MEASURED_PEAKS.json lacks (bench.py times them with
 * CUDA events).  mode 0: FP32 FMA, blocks x 256 threads x iters x 128 FMA; mode 1: MUFU ex2, blocks x 256
 * threads x iters x 64 ex2.  scratch: >= 4 bytes of device memory. */
int sgpmp_probe(int32_t mode, int32_t blocks, int32_t iters, void* scratch, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* STOCH_GPMP_B200_H */
