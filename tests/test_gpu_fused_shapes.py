"""The fused iteration kernel at the launch shapes the benchmark and the planner run, against the fp64 oracle.

Which kernel a launch runs is decided at run time (sgpmp_iterate.cu launch_iterate, sgpmp_iterate_split.cu launch_split_chain /
launch_state_only) from the grid size, S and the cost list.  Every case here names the kernel it means to test as a regex written
out by hand, and a torch.profiler probe checks that this kernel really ran: when a later change moves a shape to another kernel,
the test says so instead of silently testing something else.

For each shape of the role-split kernel (Panda: state warps + link warps; planar: state warps only), five checks:
  1. the in-kernel Philox stream gives bit-identical pass-1 costs to the same launch fed the eps the sampling kernel emits for the
     same (seed, draw, problem);
  2. that injected-eps launch matches oracle.planner.iterate (fp64) on three problems: costs to TOL_F32, weights / grad / means
     against oracle.update fed the kernel's own costs;
  3. n_iters = 4 in one launch equals four single-iteration launches bit for bit (the ring and result-barrier phases carry over
     across sweeps and iterations);
  4. the outputs requested do not change the means;
  5. the same launch twice is bit-identical.
"""
import contextlib
import re

import numpy as np
import pytest
import torch

from oracle import planner as OP
from oracle import prior as P
from oracle import update as U
from oracle.make_golden import shipped_target_H
from stoch_gpmp_b200 import scenarios as SC

from helpers import TOL_F32, from_sminor, rel

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------ dispatch probe
@contextlib.contextmanager
def kernels_launched():
    """Names of the CUDA kernels launched inside the block (torch.profiler / CUPTI; demangled, e.g.
    'sgpmp::iterate_split_kernel<7, 1, 8, 8>(...)').  The list is filled when the block ends.  A block that launched work from
    libsgpmp.so but recorded no sgpmp:: kernel means the profiler does not see the library's launches: that is an error, never a
    skip, because every dispatch assertion would then be empty.  (Seen on a B200 with torch 2.11: after the low-latency form's
    launches in the same process the profiler recorded no kernels at all.  The tests that use the probe run before those.)"""
    from torch.profiler import ProfilerActivity, profile
    names = []
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        yield names
        torch.cuda.synchronize()
    names.extend(sorted({e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}))
    if not any("sgpmp::" in nm for nm in names):
        raise AssertionError("torch.profiler recorded no sgpmp:: kernel (recorded: %s); the dispatch probe is blind" % names)


@contextlib.contextmanager
def expect_kernel(regex):
    """Assert that a kernel whose demangled name matches `regex` ran inside the block."""
    with kernels_launched() as names:
        yield names
    hit = [nm for nm in names if re.search(regex, nm)]
    assert hit, "expected a kernel matching %r; launched: %s" % (regex, names)
    print("kernel:", hit[0].split("(")[0])


def _ops():
    from stoch_gpmp_b200 import ops
    return ops


def _k():
    import test_gpu_kernels
    return test_gpu_kernels


# ------------------------------------------------------------------------------------------------ case builders
def _noisy_means(start, goals, dt, T, n, rs, noise):
    """P.const_vel_trajectories [G*K, T, d] plus N(0, noise^2) on the interior steps (start and goal rows stay exact)."""
    mu = P.const_vel_trajectories(start, goals, dt, T, n, 1).reshape(goals.shape[0], T, 2 * n)
    inner = ((np.arange(T) > 0) & (np.arange(T) < T - 1))[None, :, None]
    return mu + noise * rs.randn(*mu.shape) * inner


# Cost sigmas of the Panda matrix.  The sampling sigmas are PANDA_SIGMAS and the start / GP / goal-prior cost sigmas PANDA_COST.
# With PANDA_COST's sigma_coll = 0.01 the GP factor (~1e10 per sample) is 4e5 times the obstacle term (measured on case c), so a
# 1e-5 check on the total would not see a wrong collision term: the obstacle and self-collision sigmas are tightened until those
# terms are 1e-2 .. 2e-1 of the cost.  The EE goal keeps the shipped sigma (7e-5, 2e-2 .. 4e-2 of the cost).
PANDA_COLL_SIGMA = 1e-4
PANDA_SELF = (0.03, 1e-3)      # (margin, sigma): the shipped margin
# soft regime (bench.py soft_regime): sampling 4 / 4 / 0.5, cost 0.5 / 0.5, coll 0.3, start and goals x 0.05 -> many live weights
SOFT_SIGMAS = dict(sigma_start_init=0.5, sigma_goal_init=0.5, sigma_gp_init=0.8, sigma_start_sample=4.0, sigma_goal_sample=4.0,
                   sigma_gp_sample=0.5)


def panda_case(dev, B, G, S, T, O, selfc=False, ee=False, shared_spheres=False, sigma_coll=PANDA_COLL_SIGMA, soft=False,
               temperature=1.0, noise=0.02, seed=0):
    """Panda (PandaFK, RBF spheres, no interpolation: the structured path) fp32.  Returns (spec_of(b), sh, desc, tab, mu0, step)."""
    dtype = torch.float32
    n, d, dt = 7, 14, 0.05
    start, goals, spheres = SC.panda_batch(B, G, O, seed0=seed)
    if shared_spheres:
        spheres = np.array(SC.panda_spheres(O, seed))[None]
    step = 0.1
    cost = dict(cost_sigma_start=SC.PANDA_COST['sigma_start'], cost_sigma_gp=SC.PANDA_COST['sigma_gp'],
                sigma_goal_prior=SC.PANDA_COST['sigma_goal_prior'], sigma_coll=sigma_coll)
    sig = SC.PANDA_SIGMAS
    if soft:
        start, goals = 0.05 * start, 0.05 * goals
        cost = dict(cost_sigma_start=0.5, cost_sigma_gp=0.5, sigma_goal_prior=20., sigma_coll=0.3)
        sig, step = SOFT_SIGMAS, 0.5
    base = dict(n_dof=n, T=T, dt=dt, G=G, K=1, S=S, temperature=temperature, step_size=step, start=start[0], **cost, **sig)
    if selfc:
        base.update(self_margin=PANDA_SELF[0], sigma_self=PANDA_SELF[1])
    if ee:
        base.update(ee_target=shipped_target_H(), sigma_ee_goal=7e-5, ee_w_pos=1., ee_w_rot=1., ee_square=True)

    def spec_of(b):
        return dict(base, goals=goals[b], spheres=spheres[0 if shared_spheres else b])

    tab = _k()._tables(dict(base, goals=goals[0]), dev)
    _, low = _k()._lowered(dict(base, goals=goals, spheres=spheres[0]), dev, dtype, B=B)
    desc = low.desc(temperature, torch.tensor(spheres, device=dev, dtype=dtype).contiguous())
    rs = np.random.RandomState(seed + 1)
    mu0 = np.stack([_noisy_means(start[b], goals[b], dt, T, n, rs, noise) for b in range(B)])
    mu0 = torch.tensor(mu0, device=dev, dtype=dtype).contiguous()
    sh = _ops().make_shape(B, G, 1, S, T, n, dtype)
    return spec_of, sh, (desc, low), tab, mu0, step


def rect_map(seed, H=200):
    """A 20 m x 20 m occupancy grid (0.1 m cells) of 15 random rectangles; overlaps count 2 or 3."""
    rs = np.random.RandomState(seed)
    m = np.zeros((H, H))
    for _ in range(15):
        x0, y0 = rs.randint(25, 175, 2)
        w, h = rs.randint(10, 30, 2)
        m[y0:y0 + h, x0:x0 + w] += 1
    return m


def planar_case(dev, B, G, S, T, n, maps="u8", seed=0):
    """State-only form: n DoF, CostGP + CostGoalPrior (+ occupancy map on q0, q1) with PLANAR_SIGMAS / PLANAR_COST (the map term
    dominates), fp32.  maps: None (no obstacle cost), 'u8' (one integer map: the byte copy), 'float' (one map with
    non-integer values: the float gather), 'per_problem' (map_of_problem: two maps, alternating over the problems)."""
    from stoch_gpmp_b200.costs.cost_functions import CostCollision, CostComposite, CostGP, CostGoalPrior
    from stoch_gpmp_b200.envs.occupancy import ObstacleMap
    dtype = torch.float32
    ta = dict(device=dev, dtype=dtype)
    d, dt = 2 * n, 0.02
    st2, gl2 = SC.planar_batch(B, G, seed0=seed)
    start = np.zeros((B, d))
    goals = np.zeros((B, G, d))
    start[:, :2], goals[:, :, :2] = st2[:, :2], gl2[:, :, :2]
    start[:, 2:n], goals[:, :, 2:n] = 0.5, -0.5
    pc = SC.PLANAR_COST
    cost = dict(cost_sigma_start=pc['sigma_start'], cost_sigma_gp=pc['sigma_gp'], sigma_goal_prior=pc['sigma_goal_prior'],
                sigma_coll=pc['sigma_coll'] if maps else None)
    base = dict(n_dof=n, T=T, dt=dt, G=G, K=1, S=S, temperature=1.0, step_size=0.5, **cost, **SC.PLANAR_SIGMAS)
    grids = []
    if maps:
        grids = [rect_map(seed)] if maps != "per_problem" else [rect_map(seed), rect_map(seed + 1)]
        if maps == "float":
            grids = [g * 0.37 for g in grids]
    map_of = (lambda b: grids[b % len(grids)]) if grids else None

    def spec_of(b):
        s = dict(base, start=start[b], goals=goals[b])
        if grids:
            s.update(map=map_of(b), map_cell_size=0.1, map_origin=(100, 100))
        return s

    cl = [CostGP(n, T, torch.tensor(start, **ta), dt, dict(sigma_start=pc['sigma_start'], sigma_gp=pc['sigma_gp']), ta),
          CostGoalPrior(n, T, multi_goal_states=torch.tensor(goals, **ta), num_particles_per_goal=1, num_samples=S,
                        sigma_goal_prior=pc['sigma_goal_prior'], tensor_args=ta)]
    if grids:
        fields = []
        for b in range(B if maps == "per_problem" else 1):
            om = ObstacleMap([20, 20], 0.1, tensor_args=ta)
            om.map = map_of(b).copy()
            fields.append(om)
        cl.append(CostCollision(n, T, field=fields if maps == "per_problem" else fields[0], sigma_coll=pc['sigma_coll']))
    low = CostComposite(n, T, cl, tensor_args=ta).lower(B, G, dev, dtype)
    if maps == "u8":
        assert low.map_u8 is not None
    elif maps == "float":
        assert low.map_u8 is None
    elif maps == "per_problem":
        assert low.map_index is not None
    desc = low.desc(1.0, None)
    tab = _k()._tables(dict(base, goals=goals[0]), dev)
    rs = np.random.RandomState(seed + 1)
    mu0 = np.stack([_noisy_means(start[b], goals[b], dt, T, n, rs, 0.3) for b in range(B)])
    mu0 = torch.tensor(mu0, device=dev, dtype=dtype).contiguous()
    sh = _ops().make_shape(B, G, 1, S, T, n, dtype)
    return spec_of, sh, (desc, low), tab, mu0, 0.5


# ------------------------------------------------------------------------------------------------ the five checks
SEED, DRAW = 7, 3


def five_checks(case, kernel, claims=(), cost_tol=TOL_F32, problems=None):
    """Runs checks 1-5 of the module docstring on a case from panda_case / planar_case; `kernel` is the regex of the kernel
    every in-kernel-RNG launch must run.  `claims`: cost terms the case is meant to cover; each must be > 1e-3 of the cost
    (without the IS term) on the oracle's breakdown, or the case would not test it."""
    spec_of, sh, (desc, _low), tab, mu0, step = case
    ops = _ops()
    B = sh.B
    it = lambda mu, n_it, draw0, **kw: ops.iterate(sh, desc, tab, step, n_it, mu, seed=SEED, draw0=draw0, **kw)
    keys = ("means_pre", "samples", "costs", "weights", "grad")

    # 5. determinism, and the reference run of check 3: four iterations in one launch, every output
    runs = []
    for rep in range(2):
        mu = mu0.clone()
        with expect_kernel(kernel):
            out = it(mu, 4, DRAW, want_samples=True)
        runs.append((mu, out))
    (mu4, o4), (mu4b, o4b) = runs
    assert torch.equal(mu4, mu4b), "same launch twice: means differ"
    for k in keys:
        assert torch.equal(o4[k], o4b[k]), "same launch twice: %s differs" % k

    # 3. four single-iteration launches with draw0 + i
    mu = mu0.clone()
    first = None
    with expect_kernel(kernel):
        for i in range(4):
            o1 = it(mu, 1, DRAW + i, want_samples=(i == 3))
            if i == 0:
                first = o1
    assert torch.equal(mu, mu4), "n_iters=4 in one launch != 4 launches: means"
    for k in keys:
        assert torch.equal(o1[k], o4[k]), "n_iters=4 in one launch != 4 launches: %s" % k

    # 4. no outputs requested: same means
    mu = mu0.clone()
    with expect_kernel(kernel):
        it(mu, 4, DRAW, want_samples=False, want_costs=False, want_weights=False, want_grad=False, want_means_pre=False)
    assert torch.equal(mu, mu4), "the outputs requested changed the means"

    # 1. in-kernel stream == the sampling kernel's eps injected, bit for bit (normal_pair_f2 and normal_pair<float> form the same
    #    products, sgpmp_rng.cuh); the eps-injected launch always runs the role-split kernel
    _, eps = ops.sample(sh, tab, mu0, seed=SEED, draw=DRAW, want_eps=True)
    mu_e = mu0.clone()
    with expect_kernel(kernel):
        oe = ops.iterate(sh, desc, tab, step, 1, mu_e, eps_in=eps.unsqueeze(0).contiguous(), want_samples=True)

    # 2. the fp64 oracle on the injected-eps launch (before check 1's assertion: a wrong cost term fails here by name)
    eps_np = from_sminor(eps.cpu().numpy()).astype(np.float64)
    mu0_np = mu0.cpu().numpy().astype(np.float64)
    costs, w_k = oe["costs"].cpu().numpy(), oe["weights"].cpu().numpy()
    grad_k, mu_k, xs_k = oe["grad"].cpu().numpy(), mu_e.cpu().numpy(), from_sminor(oe["samples"].cpu().numpy())
    for b in (problems if problems is not None else sorted({0, B // 2, B - 1})):
        spec = spec_of(b)
        r = OP.iterate(spec, mu0_np[b], eps_np[b])
        wo_is = np.abs(r["costs"] - r["terms"]["is"]).max()
        shares = {k: float(np.abs(v).max() / wo_is) for k, v in r["terms"].items()}
        e_c = rel(costs[b], r["costs"])
        mp, grad, w = U.update(mu0_np[b], r["samples"], costs[b].astype(np.float64), spec["temperature"], spec["step_size"])
        e_w, e_g, e_m = float(np.abs(w_k[b] - w).max()), rel(grad_k[b], grad), rel(mu_k[b], mp)
        print("problem %d: costs %.1e samples %.1e weights %.1e grad %.1e means %.1e | live weights %d | shares %s" % (
            b, e_c, rel(xs_k[b], r["samples"]), e_w, e_g, e_m, int((w > 0).sum()),
            " ".join("%s %.0e" % kv for kv in sorted(shares.items()))))
        for term in claims:
            assert shares[term] > 1e-3, "the %s term is %.1e of the cost here: this case does not test it" % (term, shares[term])
        assert rel(xs_k[b], r["samples"]) < TOL_F32
        assert e_c < cost_tol
        assert e_w < 1e-5
        assert e_g < 2e-5
        assert e_m < 1e-6
    assert torch.equal(oe["costs"], first["costs"]), "in-kernel Philox != injected eps: pass-1 costs (max rel %.2e)" % (
        float((oe["costs"] - first["costs"]).abs().max() / first["costs"].abs().max()))
    assert torch.equal(oe["weights"], first["weights"])
    return oe


# ------------------------------------------------------------------------------------------------ role-split Panda kernel
# (B, G, S, T, O, self, EE, shared spheres, expected kernel, claimed terms)
PANDA_CASES = {
    # 1+1 warps, one ragged sweep, 3 ring stages; OC=8; self-collision (CHAIN 2)
    "a": ((2, 2, 17, 13, 8, True, False, False), r"iterate_split_kernel<7, ?2, ?1, ?1>", ("coll", "self")),
    # 2+2 warps, one ragged sweep, one stage (T=2, the shortest horizon); OC=4; EE goal
    "b": ((2, 2, 50, 2, 4, False, True, False), r"iterate_split_kernel<7, ?1, ?2, ?2>", ("coll", "ee")),
    # 4+4 warps, 2 sweeps (72 samples in the last), 13 stages; the shipped list: 5 spheres + self + EE
    "c": ((38, 4, 200, 64, 5, True, True, False), r"iterate_split_kernel<7, ?2, ?4, ?4>", ("coll", "self", "ee")),
    # 8+8 warps, 2 sweeps: the C4 per-problem shape at the 8-GPU shard size, spheres per problem
    "d": ((38, 4, 512, 64, 5, False, False, False), r"iterate_split_kernel<7, ?1, ?8, ?8>", ("coll",)),
    # 8+8 warps, 2 sweeps (44 in the last), 16 shared spheres (the limit; the run-time sphere loop)
    "e": ((50, 3, 300, 11, 16, False, False, True), r"iterate_split_kernel<7, ?1, ?8, ?8>", ("coll",)),
}


@pytest.mark.parametrize("name", sorted(PANDA_CASES))
def test_split_panda_shapes(name, cuda):
    (B, G, S, T, O, selfc, ee, shared), kernel, claims = PANDA_CASES[name]
    # case b: one collision step (T=2) in free space; the obstacle sigma is tightened further so that the term is visible
    sigma_coll = 1e-6 if name == "b" else PANDA_COLL_SIGMA
    case = panda_case(cuda, B, G, S, T, O, selfc=selfc, ee=ee, shared_spheres=shared, sigma_coll=sigma_coll)
    five_checks(case, kernel, claims)


def test_split_panda_soft_weights(cuda):
    """Soft regime (bench.py soft_regime's sigmas), 4+4 warps, 2 sweeps.  The costs without the IS term spread over ~1.3e3 per
    particle; at temperature 200 every sample keeps a live weight (oracle, random eps), so pass 2 sums many non-zero weights."""
    case = panda_case(cuda, 38, 4, 160, 32, 5, soft=True, temperature=200., noise=0.0)
    # costs: 2.5e-5 measured (problems 0 / 19 / 37: 2.5e-5 / 1.6e-5 / 1.8e-5; K3 on the same samples 2.6e-5 / 1.9e-5 / 2.7e-5).  The
    # IS term limits it: tau x^T P mu is formed in fp32 from terms that cancel, its error is 2.4e-4 of itself and 2.7e-5 of the
    # largest cost (every other term <= 9e-6).  3e-5 is the floor test_fused_iteration_matches_reference allows the soft goldens.
    oe = five_checks(case, r"iterate_split_kernel<7, ?1, ?4, ?4>", ("coll",), cost_tol=3e-5)
    live = (oe["weights"] > 1e-6).sum(-1)
    assert int(live.min()) >= 8, "pass 2 saw at most %d live weights" % int(live.min())


def _grid_equals_shards(cuda, S, T, samples):
    """The 1-GPU benchmark grid (1,537 problems x 4 goals: 6,148 CTAs, 4+4 warps) in one launch against its first and last 38
    problems launched alone with problem_gid0 (8+8 warps).  A sample's arithmetic does not depend on the CTA shape: per-sample
    costs (and samples, when `samples`) are bit-identical; weights, grad and means agree to the rounding of the block sums."""
    B, G = 1537, 4
    ops = _ops()
    spec_of, sh, (desc, _), tab, mu0, step = panda_case(cuda, B, G, S, T, 5)
    mu = mu0.clone()
    with expect_kernel(r"iterate_split_kernel<7, ?1, ?4, ?4>"):
        out = ops.iterate(sh, desc, tab, step, 1, mu, seed=SEED, draw0=DRAW, want_samples=samples, want_means_pre=False)
    _, goals, spheres = SC.panda_batch(B, G, 5, seed0=0)
    for lo in (0, B - 38):
        hi = lo + 38
        base = spec_of(lo)
        _, lowp = _k()._lowered(dict(base, goals=goals[lo:hi], spheres=spheres[0]), cuda, torch.float32, B=38)
        descp = lowp.desc(1.0, torch.tensor(spheres[lo:hi], device=cuda, dtype=torch.float32).contiguous())
        shp = ops.make_shape(38, G, 1, S, T, 7, torch.float32, problem_gid0=lo)
        mup = mu0[lo:hi].clone()
        with expect_kernel(r"iterate_split_kernel<7, ?1, ?8, ?8>"):
            op = ops.iterate(shp, descp, tab, step, 1, mup, seed=SEED, draw0=DRAW, want_samples=samples, want_means_pre=False)
        assert torch.equal(out["costs"][lo:hi], op["costs"]), "problems %d..%d: per-sample costs differ" % (lo, hi - 1)
        if samples:
            assert torch.equal(out["samples"][lo:hi], op["samples"]), "problems %d..%d: samples differ" % (lo, hi - 1)
        assert float((out["weights"][lo:hi] - op["weights"]).abs().max()) < 1e-6
        assert float((out["grad"][lo:hi] - op["grad"]).abs().max() / op["grad"].abs().max()) < 1e-5
        assert float((mu[lo:hi] - mup).abs().max() / mup.abs().max()) < 1e-6


def test_split_panda_bench_grid_equals_shards(cuda):
    """Case f: _grid_equals_shards at the benchmark's shape (S=512, T=64: 4 sweeps), per-sample costs."""
    _grid_equals_shards(cuda, 512, 64, samples=False)


def test_split_panda_cta_shapes_agree(cuda):
    """_grid_equals_shards at a short horizon (S=256, T=8), where the grid's samples (0.7 GB) fit: costs AND samples of the 4+4
    and the 8+8 warp shapes are bit-identical."""
    _grid_equals_shards(cuda, 256, 8, samples=True)


# ------------------------------------------------------------------------------------------------ state-only form
@pytest.mark.parametrize("S,na", [(20, 1), (40, 2), (100, 4)])
@pytest.mark.parametrize("n", [2, 3, 4, 6])
def test_split_state_only_shapes(n, S, na, cuda):
    """n DoF x 1 / 2 / 4 state warps (S = 20 / 40 / 100: one ragged sweep), T = 24 (two 16-step stages), the byte map."""
    case = planar_case(cuda, 3, 2, S, 24, n, maps="u8")
    five_checks(case, r"iterate_split_kernel<%d, ?0, ?%d, ?0>" % (n, na), ("coll",))


@pytest.mark.parametrize("n,S,maps", [(2, 100, "float"), (6, 40, "float"), (3, 20, "per_problem"), (4, 100, "per_problem")])
def test_split_state_only_map_forms(n, S, maps, cuda):
    """The float gather (a map with non-integer values) and two maps chosen per problem (map_of_problem)."""
    na = 4 if S > 64 else (2 if S > 32 else 1)
    case = planar_case(cuda, 4, 2, S, 24, n, maps=maps)
    five_checks(case, r"iterate_split_kernel<%d, ?0, ?%d, ?0>" % (n, na), ("coll",))


def test_split_state_only_c2_shape(cuda):
    """The C2 per-problem shape at 152 particles (38 problems x 4 goals, S=256, T=64): 4 state warps, 2 sweeps, two maps."""
    case = planar_case(cuda, 38, 4, 256, 64, 2, maps="per_problem")
    five_checks(case, r"iterate_split_kernel<2, ?0, ?4, ?0>", ("coll",))


@pytest.mark.parametrize("maps", [None, "u8"])
@pytest.mark.parametrize("S", [1, 3, 4])
@pytest.mark.parametrize("n", [2, 3])
def test_split_state_only_t2_smallest_grid(n, S, maps, cuda):
    """T=2 with S <= 4: the block phases alone need 64 or 80 bytes of the union region, less than the 32 floats of start-up
    staging that share it (launch_split_cfg sizes the region for both).  S=1: one weight of 1."""
    case = planar_case(cuda, 3, 2, S, 2, n, maps=maps)
    oe = five_checks(case, r"iterate_split_kernel<%d, ?0, ?1, ?0>" % n)
    if S == 1:
        assert torch.equal(oe["weights"], torch.ones_like(oe["weights"]))


# ------------------------------------------------------------------------------------------------ planner level
@pytest.mark.parametrize("workload,kernel", [("panda", r"iterate_split_kernel<7, ?1, ?8, ?8>"),
                                             ("planar", r"iterate_split_kernel<2, ?0, ?4, ?0>")], ids=["panda", "planar"])
def test_optimize_many_iterations_equals_single_calls(workload, kernel, cuda):
    """StochGPMPBatch at the benchmark's per-problem shapes, 38 problems (the role-split kernel): optimize(opt_iters=5) — all
    iterations in one launch — equals five optimize(opt_iters=1) calls bit for bit, means and last costs.  The examples' plans
    ("one call of 501 iterations") rely on this."""
    import bench
    w = bench.workload(workload, 38)
    obs = {"obstacle_spheres": torch.tensor(w["spheres"], dtype=torch.float32, device=cuda)} if w["spheres"] is not None else {}
    one, many = bench.build_planner(w, 38, cuda), bench.build_planner(w, 38, cuda)
    with expect_kernel(kernel):
        r1 = one.optimize(opt_iters=5, return_samples=False, **obs)
    with expect_kernel(kernel):
        for _ in range(5):
            r5 = many.optimize(opt_iters=1, return_samples=False, **obs)
    assert torch.equal(one.particle_means, many.particle_means)
    assert torch.equal(r1[4], r5[4])
    assert torch.equal(r1[0], r5[0]) and torch.equal(r1[5], r5[5])
