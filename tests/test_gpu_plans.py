"""GPU: StochGPMPBatch.best_plans / sgpmp_select_plans — the collision check of the final means between and at their support
states, and the choice of each problem's plan — against the numpy oracle (oracle/plans.py)."""
import math
import random

import numpy as np
import pytest
import torch

from oracle import fk as OFK
from oracle import plans as OPL

from helpers import rel

pytestmark = pytest.mark.gpu

DT = 0.05


def _target_H(ta):
    c, s = math.cos(-math.pi), math.sin(-math.pi)
    H = torch.eye(4, dtype=torch.float64)
    H[:3, :3] = torch.tensor([[c, -s, 0.], [s, c, 0.], [0., 0., 1.]], dtype=torch.float64) @ \
        torch.tensor([[c, 0., s], [0., 1., 0.], [-s, 0., c]], dtype=torch.float64)
    H[:3, 3] = torch.tensor([.3, .3, .3], dtype=torch.float64)
    return H.to(**ta).unsqueeze(0)


def _panda(dev, dtype, B, T=16, G=2, K=2, S=64, interp=0, iters=3, batched=True, spheres=None, goals=None, cost_list=None):
    """The shipped Panda cost list (examples/panda_environment.py) over B problems with their own goals and spheres."""
    from stoch_gpmp_b200 import scenarios as sc
    from stoch_gpmp_b200.costs.cost_functions import CostCollision, CostComposite, CostGP, CostGoal, CostGoalPrior
    from stoch_gpmp_b200.costs.fields import EESE3DistanceField, LinkDistanceField, LinkSelfDistanceField
    from stoch_gpmp_b200.planner import StochGPMP, StochGPMPBatch
    from stoch_gpmp_b200.robots import PandaFK
    ta = dict(device=dev, dtype=dtype)
    start, g, sp = sc.panda_batch(B, G=G, O=5, seed0=3)
    goals = g if goals is None else goals
    spheres = sp if spheres is None else spheres
    n = 7
    s_t, g_t = torch.tensor(start, **ta), torch.tensor(goals, **ta)
    if not batched:
        s_t, g_t = s_t[0], g_t[0]
    cl = [CostGP(n, T, s_t, DT, dict(sigma_start=0.0001, sigma_gp=0.0007), ta),
          CostGoalPrior(n, T, multi_goal_states=g_t, num_particles_per_goal=K, num_samples=S, sigma_goal_prior=20., tensor_args=ta),
          CostCollision(n, T, field=LinkSelfDistanceField(margin=0.03, tensor_args=ta), sigma_coll=0.01),
          CostCollision(n, T, field=LinkDistanceField(num_interpolate=interp, tensor_args=ta), sigma_coll=0.01),
          CostGoal(n, T, field=EESE3DistanceField(_target_H(ta), tensor_args=ta), sigma_goal=0.00007)]
    if cost_list is not None:
        cl = cl + cost_list
    cost = CostComposite(n, T, cl, FK=PandaFK(), tensor_args=ta)
    cls = StochGPMPBatch if batched else StochGPMP
    pl = cls(num_particles_per_goal=K, num_samples=S, traj_len=T, opt_iters=iters, dt=DT, n_dof=n, step_size=0.1, temperature=1.,
             start_state=s_t, multi_goal_states=g_t, initial_particle_means='const_vel', cost=cost, seed=0, tensor_args=ta,
             **sc.PANDA_SIGMAS)
    obs = {'obstacle_spheres': torch.tensor(spheres if batched else spheres[:1], **ta)}
    return pl, obs, np.asarray(spheres, dtype=np.float64)


def _check_selection(res, oracle_clear, margin, tol):
    """particle / collision_free equal the oracle's rule on the kernel's own costs; problems with a particle within tol of the
    margin are left out (their feasibility is decided by the last bits)."""
    costs = res.particle_costs.cpu().numpy()
    hits = res.particle_hits.cpu().numpy()
    keep = ~(np.abs(oracle_clear - margin) < tol).any(1)
    assert keep.sum() >= 0.75 * len(keep)
    p, ok = OPL.select(costs, oracle_clear, hits, margin)
    assert np.array_equal(res.particle.cpu().numpy()[keep], p[keep])
    assert np.array_equal(res.collision_free.cpu().numpy()[keep], ok[keep])
    return keep


CASES = [(torch.float64, 0, 0), (torch.float64, 3, 0), (torch.float64, 8, 2),
         (torch.float32, 0, 0), (torch.float32, 3, 2), (torch.float32, 8, 0)]


@pytest.mark.parametrize("dtype,n_interp,link_interp", CASES, ids=lambda v: str(v).replace("torch.", ""))
def test_panda_matches_oracle(cuda, dtype, n_interp, link_interp):
    from stoch_gpmp_b200 import ops
    from stoch_gpmp_b200.robots import PandaFK
    f64 = dtype == torch.float64
    B, T = 24, 16
    pl, obs, spheres = _panda(cuda, dtype, B, T=T, interp=link_interp)
    pl.optimize(**obs)
    means = pl.particle_means.clone()
    mu = means.cpu().numpy().astype(np.float64)
    # oracle clearance at margin 0 decides the margin: the median particle, so that both outcomes occur
    oc = np.stack([OPL.clearance(mu[b], spheres[b], DT, n_interp, link_interp) for b in range(B)])
    margin = float(np.median(oc))
    res = pl.best_plans(n_interp=n_interp, margin=margin, **obs)
    P = (T - 1) * (n_interp + 1) + 1
    assert tuple(res.dense_plan.shape) == (B, P, 14) and res.dense_dt == DT / (n_interp + 1)
    assert torch.equal(pl.particle_means, means)                           # nothing changes the planner's state
    clear = res.particle_clearance.cpu().numpy()
    assert np.abs(clear - oc).max() < (1e-12 if f64 else 1e-5)
    assert np.array_equal(res.particle_hits.cpu().numpy(), np.zeros((B, 4), np.int32))
    _check_selection(res, oc, margin, 1e-5)
    # the plan is the chosen mean bit for bit; the dense plan holds it at every (n_interp+1)-th state
    idx = res.particle
    assert torch.equal(res.plan, means[torch.arange(B, device=cuda), idx])
    assert torch.equal(res.dense_plan[:, ::n_interp + 1], res.plan)
    assert rel(res.dense_plan.cpu().numpy(), OPL.dense(res.plan.cpu().numpy(), DT, n_interp)) < (1e-12 if f64 else 1e-6)
    assert torch.equal(res.cost, res.particle_costs.gather(1, idx[:, None])[:, 0])
    assert torch.equal(res.clearance, res.particle_clearance.gather(1, idx[:, None])[:, 0])
    # the ranking cost is the cost kernel on the means without the IS term, bit for bit
    desc = pl._lowered.desc(0.0, obs['obstacle_spheres'])
    want = ops.cost(pl._shape(S=1), desc, None, means.unsqueeze(-1).contiguous(), None)[..., 0]
    assert torch.equal(res.particle_costs, want)
    if n_interp == 0 and link_interp == 0:
        # the hand-written check of the shipped example (link origins by ops.fk_link_positions, torch distances), states t >= 1
        q = means[:, :, 1:, :7].reshape(-1, 7).contiguous()
        pos = ops.fk_link_positions(PandaFK(), q).reshape(B, -1, 11, 3)
        sph = obs['obstacle_spheres']
        dist = (pos[:, :, :, None, :] - sph[:, None, None, :, :3]).norm(dim=-1) - sph[:, None, None, :, 3]
        old = dist.reshape(B, 4, -1).amin(-1)
        assert (res.particle_clearance - old).abs().max().item() < 1e-6


def _planar(dev, dtype, B, maps, T=16, G=2, K=2, S=64, iters=3):
    from stoch_gpmp_b200 import scenarios as sc
    from stoch_gpmp_b200.costs.cost_functions import CostCollision, CostComposite, CostGP, CostGoalPrior
    from stoch_gpmp_b200.planner import StochGPMPBatch
    ta = dict(device=dev, dtype=dtype)
    start, goals = sc.planar_batch(B, G=G, seed0=5)
    s_t, g_t = torch.tensor(start, **ta), torch.tensor(goals, **ta)
    c = sc.PLANAR_COST
    cost = CostComposite(2, T, [CostGP(2, T, s_t, 0.02, dict(sigma_start=c['sigma_start'], sigma_gp=c['sigma_gp']), ta),
                                CostGoalPrior(2, T, multi_goal_states=g_t, num_particles_per_goal=K, num_samples=S,
                                              sigma_goal_prior=c['sigma_goal_prior'], tensor_args=ta),
                                CostCollision(2, T, field=maps if B > 1 else maps[0], sigma_coll=c['sigma_coll'])], tensor_args=ta)
    return StochGPMPBatch(num_particles_per_goal=K, num_samples=S, traj_len=T, opt_iters=iters, dt=0.02, n_dof=2, step_size=0.5,
                          temperature=1., start_state=s_t, multi_goal_states=g_t, initial_particle_means='const_vel', cost=cost,
                          seed=0, tensor_args=ta, **sc.PLANAR_SIGMAS)


def _maps(B, dtype, scale=1.0):
    from stoch_gpmp_b200.envs.map_generator import generate_obstacle_map
    out = []
    for b in range(B):
        random.seed(200 + b)
        np.random.seed(200 + b)
        m = generate_obstacle_map(map_dim=[20, 20], cell_size=0.1, random_gen=True, num_obst=15, rand_limits=[[-7.5, 7.5], [-7.5, 7.5]],
                                  rand_rect_shape=[2, 2], tensor_args=dict(device='cpu', dtype=dtype))[0]
        m.map = m.map * scale
        out.append(m)
    return out


@pytest.mark.parametrize("byte_map", [True, False], ids=["byte_map", "float_map"])
def test_planar_hits_match_oracle(cuda, byte_map):
    B, T, m = 12, 16, 4
    maps = _maps(B, torch.float64, 1.0 if byte_map else 0.5)          # counts * 0.5 are not bytes: the float map is gathered
    pl = _planar(cuda, torch.float64, B, maps, T=T)
    assert (pl._lowered.map_u8 is not None) == byte_map
    pl.optimize()
    mu = pl.particle_means.cpu().numpy()
    res = pl.best_plans(n_interp=m)
    # states within 1e-9 of a cell edge may round either way between the two evaluation orders: there are none here
    xy = OPL.dense(mu, 0.02, m)[..., 1:, :2] * 10.0
    assert np.abs(xy - np.round(xy)).min() > 1e-9
    want = np.stack([OPL.hits(mu[b], maps[b].map, 0.1, maps[b].origin_xi, maps[b].origin_yi, 0.02, m) for b in range(B)])
    got = res.particle_hits.cpu().numpy()
    assert np.array_equal(got, want)
    assert got.any() and (got == 0).any()
    assert torch.isinf(res.particle_clearance).all()
    p, ok = OPL.select(res.particle_costs.cpu().numpy(), np.full(got.shape, np.inf), want, 0.0)
    assert np.array_equal(res.particle.cpu().numpy(), p) and np.array_equal(res.collision_free.cpu().numpy(), ok)
    assert torch.equal(res.dense_plan[:, ::m + 1], res.plan)


def test_panda_collision_between_support_states(cuda):
    """Every support state is clear of the sphere, an interpolated state is not: collision-free at n_interp = 0 only."""
    T, dtype = 8, torch.float64
    q0 = np.array([-1.0, -0.57, 0., -2.81, 0., 3.037, 0.741])
    dq = np.zeros(7)
    dq[0] = 2.0 / (T - 1)                                 # base joint sweeps; constant velocity: the interpolation is linear in q
    mean = np.zeros((T, 14))
    mean[:, :7] = q0 + np.arange(T)[:, None] * dq
    mean[:, 7:] = dq / DT
    mid = 0.5 * (mean[3, :7] + mean[4, :7])               # middle of interval 3
    ee = lambda q: OFK.fk_all_links(np.atleast_2d(q))[:, -1, :3, 3]
    span = np.linalg.norm(ee(mean[3, :7]) - ee(mean[4, :7]))
    sphere = np.concatenate([ee(mid)[0], [0.25 * span]])[None, None]          # [1, 1, 4]
    assert OPL.clearance(mean, sphere[0], DT, 0) > 0.01
    pl, obs, _ = _panda(cuda, dtype, 1, T=T, G=1, K=1, S=16, spheres=sphere, goals=np.tile(mean[-1], (1, 1, 1)))
    pl.particle_means = torch.tensor(mean[None, None], device=cuda, dtype=dtype)
    r0 = pl.best_plans(n_interp=0, **obs)
    assert bool(r0.collision_free[0]) and r0.clearance[0].item() > 0.01
    for m in (1, 2, 3, 8):
        r = pl.best_plans(n_interp=m, **obs)
        assert not bool(r.collision_free[0]), m
        assert abs(r.clearance[0].item() - OPL.clearance(mean, sphere[0], DT, m)) < 1e-12


def test_planar_jump_across_a_one_cell_wall(cuda):
    from stoch_gpmp_b200.envs.occupancy import ObstacleMap
    T, dtype = 8, torch.float64
    wall = ObstacleMap(map_dim=[20, 20], cell_size=0.1)
    wall.map[:, wall.origin_xi] = 1                       # x in [0, 0.1): one cell wide, all along y
    pl = _planar(cuda, dtype, 1, [wall], T=T, G=1, K=1, S=16)
    x = -0.12 + 0.3 * (np.arange(T) - 3)                  # supports -0.12 | 0.18 straddle the wall
    mean = np.zeros((1, 1, T, 4))
    mean[..., 0], mean[..., 1], mean[..., 2] = x, 0.05, 0.3 / 0.02
    pl.particle_means = torch.tensor(mean, device=cuda, dtype=dtype)
    r0 = pl.best_plans(n_interp=0)
    assert bool(r0.collision_free[0]) and r0.particle_hits[0, 0].item() == 0
    for m in (1, 2, 3, 8):
        r = pl.best_plans(n_interp=m)
        assert not bool(r.collision_free[0]) and r.particle_hits[0, 0].item() >= 1, m
        assert r.particle_hits[0, 0].item() == OPL.hits(mean[0, 0], wall.map, 0.1, wall.origin_xi, wall.origin_yi, 0.02, m)


def test_selection_rule_edges(cuda):
    """Kernel-level: lowest-cost particle skipped when it collides, argmin with ok = 0 when none is feasible, ties to the lowest
    index, NaN never feasible."""
    from stoch_gpmp_b200 import ops
    pl, obs, spheres = _panda(cuda, torch.float64, 5, T=8, G=1, K=4, S=16, iters=1)
    pl.optimize(**obs)
    desc = pl._lowered.desc(0.0, obs['obstacle_spheres'])
    base = pl.best_plans(n_interp=2, **obs)
    clear = base.particle_clearance.cpu().numpy()
    margin = float(np.median(clear))
    assert (np.abs(clear - margin) > 1e-9).sum() >= 15
    nan = float('nan')
    costs = torch.tensor([[1., 2., 3., 4.], [5., 4., 4., 5.], [3., 1., 2., 1.], [nan, 2., 1., 3.], [1., 1., 1., 1.]],
                         device=cuda, dtype=torch.float64)
    r = ops.select_plans(pl._shape(S=1), desc, pl._means, costs, 2, margin)
    p, ok = OPL.select(costs.cpu().numpy(), clear, np.zeros_like(clear), margin)
    assert np.array_equal(r['particle'].cpu().numpy(), p) and np.array_equal(r['ok'].cpu().numpy().astype(bool), ok)
    # margin +1e3: nothing is feasible -> argmin over all (ties to the lowest index), ok = 0
    r = ops.select_plans(pl._shape(S=1), desc, pl._means, costs, 2, 1e3)
    assert r['particle'].tolist() == [0, 1, 1, 2, 0] and r['ok'].tolist() == [0] * 5
    # margin -1e3: everything with a finite cost is feasible; NaN is not
    r = ops.select_plans(pl._shape(S=1), desc, pl._means, costs, 2, -1e3)
    assert r['particle'].tolist() == [0, 1, 1, 2, 0] and r['ok'].tolist() == [1] * 5
    allnan = torch.full((5, 4), nan, device=cuda, dtype=torch.float64)
    r = ops.select_plans(pl._shape(S=1), desc, pl._means, allnan, 2, -1e3)
    assert r['particle'].tolist() == [0] * 5 and r['ok'].tolist() == [0] * 5


def test_batch_equals_single_problems(cuda):
    from stoch_gpmp_b200.gpmp import GPMP
    from stoch_gpmp_b200.planner import StochGPMPBatch
    B, T = 3, 16
    pl, obs, spheres = _panda(cuda, torch.float32, B, T=T)
    pl.optimize(**obs)
    means = pl.particle_means.clone()
    full = pl.best_plans(n_interp=5, margin=0.05, **obs)
    from stoch_gpmp_b200 import scenarios as sc
    _, goals, _ = sc.panda_batch(B, G=2, O=5, seed0=3)
    for b in range(B):
        one, o1, _ = _panda(cuda, torch.float32, 1, T=T, spheres=spheres[b:b + 1], goals=goals[b:b + 1])
        single, os_, _ = _panda(cuda, torch.float32, 1, T=T, spheres=spheres[b:b + 1], goals=goals[b:b + 1], batched=False)
        assert isinstance(one, StochGPMPBatch) and not single._batched
        one.particle_means = means[b:b + 1]
        single.particle_means = means[b]
        r1 = one.best_plans(n_interp=5, margin=0.05, **o1)
        rs = single.best_plans(n_interp=5, margin=0.05, **os_)
        for name, v in full._asdict().items():
            if name == 'dense_dt':
                assert v == r1.dense_dt == rs.dense_dt
                continue
            assert torch.equal(v[b], r1._asdict()[name][0]), name
            assert torch.equal(r1._asdict()[name][0], rs._asdict()[name]), name
    # the Gauss-Newton planner has the same means and lowered cost
    from stoch_gpmp_b200.costs.cost_functions import CostCollision, CostComposite, CostGP, CostGoalPrior
    from stoch_gpmp_b200.costs.fields import LinkDistanceField
    from stoch_gpmp_b200.robots import PandaFK
    ta = dict(device=cuda, dtype=torch.float64)
    start = torch.tensor(sc.PANDA_START, **ta)
    goal = torch.tensor(sc.panda_goals(1, 7), **ta)
    cost = CostComposite(7, T, [CostGP(7, T, start, DT, dict(sigma_start=0.001, sigma_gp=0.1), ta),
                                CostGoalPrior(7, T, multi_goal_states=goal, num_particles_per_goal=2, num_samples=1,
                                              sigma_goal_prior=0.01, tensor_args=ta),
                                CostCollision(7, T, field=LinkDistanceField(tensor_args=ta), sigma_coll=0.02)], FK=PandaFK(), tensor_args=ta)
    gp = GPMP(num_particles_per_goal=2, traj_len=T, opt_iters=2, dt=DT, n_dof=7, step_size=0.3, start_state=start,
              multi_goal_states=goal, cost=cost, initial_particle_means='const_vel', solver_params=dict(delta=1e-2, trust_region=True,
              method='inverse'), seed=0, tensor_args=ta, **sc.PANDA_SIGMAS)
    sp = torch.tensor(spheres[:1], **ta)
    gp.optimize(obstacle_spheres=sp)
    r = gp.best_plans(n_interp=4, obstacle_spheres=sp)
    assert torch.equal(r.plan, gp.particle_means[r.particle])
    assert abs(r.clearance.item() - OPL.clearance(gp.particle_means[r.particle].cpu().numpy(), spheres[0], DT, 4)) < 1e-12


def test_errors(cuda):
    from stoch_gpmp_b200 import ops
    from stoch_gpmp_b200.costs.cost_functions import CostComposite, CostGP
    pl, obs, _ = _panda(cuda, torch.float32, 2, T=8, G=1, K=2, S=16, iters=1)
    for m in (-1, 33):
        with pytest.raises(ValueError, match="n_interp"):
            pl.best_plans(n_interp=m, **obs)
    with pytest.raises(ValueError, match="margin"):
        pl.best_plans(margin=float('nan'), **obs)
    user = _panda(cuda, torch.float32, 2, T=8, G=1, K=2, S=16, iters=1,
                  cost_list=[lambda trajs, x_trajs=None, **kw: trajs[:, :, 0].sum(-1)])[0]
    assert user._lowered.custom
    with pytest.raises(NotImplementedError, match="user-defined"):
        user.best_plans(**obs)
    # a DoF count the library does not instantiate
    ta = dict(device=cuda, dtype=torch.float32)
    n, T = 9, 8
    desc = CostComposite(n, T, [CostGP(n, T, torch.zeros(2 * n, **ta), DT, dict(sigma_start=1., sigma_gp=1.), ta)]).lower(
        1, 1, cuda, torch.float32).desc(0.0)
    with pytest.raises(NotImplementedError, match="n_dof=9"):
        ops.select_plans(ops.make_shape(1, 1, 1, 1, T, n, torch.float32), desc, torch.zeros(1, 1, T, 2 * n, **ta),
                         torch.zeros(1, 1, **ta), 2, 0.0)


def test_full_c4_shape(cuda):
    """4096 problems x 4 particles, T = 64, 5 spheres each, n_interp = 8: matches the oracle on the first and last 8 problems."""
    import bench
    w = bench.workload("panda", 4096)
    pl = bench.build_planner(w, 4096, cuda)
    obs = {'obstacle_spheres': torch.tensor(w["spheres"], device=cuda, dtype=torch.float32)}
    pl.optimize(opt_iters=2, **obs)
    mu = pl.particle_means.cpu().numpy().astype(np.float64)
    res = pl.best_plans(n_interp=8, **obs)
    rows = list(range(8)) + list(range(4088, 4096))
    oc = np.stack([OPL.clearance(mu[b], w["spheres"][b], w["dt"], 8) for b in rows])
    assert np.abs(res.particle_clearance.cpu().numpy()[rows] - oc).max() < 1e-5
    sub = type(res)(*[v[rows] if isinstance(v, torch.Tensor) else v for v in res])
    _check_selection(sub, oc, 0.0, 1e-5)
    assert torch.equal(res.plan, pl.particle_means[torch.arange(4096, device=cuda), res.particle])
    assert torch.equal(res.dense_plan[:, ::9], res.plan)
