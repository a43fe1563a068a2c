"""The reference's examples/panda_environment.py on stoch_gpmp_b200 (headless, no pybullet / torch_robotics).

Same cost list and parameters as the reference script (examples/panda_environment.py:29-146): CostGP, CostGoalPrior,
self-collision, obstacle spheres and the EE SE(3) goal (CostGoal + EESE3DistanceField; SE3_distance as restated in
DESIGN.md §3).  The IK goal of pybullet is replaced by a fixed joint-space goal and the obstacle spheres are drawn
with numpy instead of the simulator.
"""
import math
import time

import numpy as np
import torch

from stoch_gpmp_b200.planner import StochGPMP
from stoch_gpmp_b200.costs.cost_functions import CostCollision, CostComposite, CostGP, CostGoal, CostGoalPrior
from stoch_gpmp_b200.costs.fields import EESE3DistanceField, LinkDistanceField, LinkSelfDistanceField
from stoch_gpmp_b200.robots import PandaFK
from stoch_gpmp_b200 import ops


if __name__ == '__main__':
    device = torch.device('cuda:0')
    tensor_args = {'device': device, 'dtype': torch.float32}
    seed = 0
    num_particles_per_goal = 5
    num_samples = 32
    num_obst = 5
    traj_len = 64
    dt = 0.05
    np.random.seed(seed)

    # world setup (examples/panda_environment.py:38-43): target_rot = Rz(-pi) Ry(-pi), target_pos = (.3, .3, .3)
    c, s = math.cos(-math.pi), math.sin(-math.pi)
    Rz = torch.tensor([[c, -s, 0.], [s, c, 0.], [0., 0., 1.]], dtype=torch.float64)
    Ry = torch.tensor([[c, 0., s], [0., 1., 0.], [-s, 0., c]], dtype=torch.float64)
    target_H = torch.eye(4, dtype=torch.float64)
    target_H[:3, :3] = Rz @ Ry
    target_H[:3, 3] = torch.tensor([.3, .3, .3], dtype=torch.float64)
    target_H = target_H.to(**tensor_args).unsqueeze(0)

    panda_fk = PandaFK()
    n_dof = panda_fk._n_dofs
    start_q = torch.tensor([0.012, -0.57, 0., -2.81, 0., 3.037, 0.741], **tensor_args)
    start_state = torch.cat((start_q, torch.zeros_like(start_q)))
    # an IK solution of the target pose (stands in for pybullet's solveInverseKinematics, examples/panda_environment.py:61)
    q_goal = torch.tensor([-0.0138, -0.4637, 0.7626, -2.5, 0.371, 2.1212, 2.8481], **tensor_args)
    multi_goal_states = torch.cat([q_goal, torch.zeros_like(q_goal)]).unsqueeze(0)

    panda_self_link = LinkSelfDistanceField(margin=0.03, tensor_args=tensor_args)
    panda_collision_link = LinkDistanceField(tensor_args=tensor_args)
    panda_goal = EESE3DistanceField(target_H, tensor_args=tensor_args)
    prior_sigmas = dict(sigma_start=0.0001, sigma_gp=0.0007)
    sigma_self, sigma_coll, sigma_goal, sigma_goal_prior = 0.01, 0.01, 0.00007, 20.
    cost_prior = CostGP(n_dof, traj_len, start_state, dt, prior_sigmas, tensor_args)
    cost_self = CostCollision(n_dof, traj_len, field=panda_self_link, sigma_coll=sigma_self)
    cost_coll = CostCollision(n_dof, traj_len, field=panda_collision_link, sigma_coll=sigma_coll)
    cost_goal_prior = CostGoalPrior(n_dof, traj_len, multi_goal_states=multi_goal_states,
                                    num_particles_per_goal=num_particles_per_goal, num_samples=num_samples,
                                    sigma_goal_prior=sigma_goal_prior, tensor_args=tensor_args)
    cost_goal = CostGoal(n_dof, traj_len, field=panda_goal, sigma_goal=sigma_goal)
    cost_composite = CostComposite(n_dof, traj_len, [cost_prior, cost_goal_prior, cost_self, cost_coll, cost_goal], FK=panda_fk)

    planner = StochGPMP(
        num_particles_per_goal=num_particles_per_goal, num_samples=num_samples, traj_len=traj_len, dt=dt, n_dof=n_dof,
        opt_iters=1, temperature=1., start_state=start_state, multi_goal_states=multi_goal_states, cost=cost_composite,
        step_size=0.1, sigma_start_init=0.0001, sigma_goal_init=0.1, sigma_gp_init=0.8, sigma_start_sample=0.001,
        sigma_goal_sample=0.07, sigma_gp_sample=0.1, seed=seed, tensor_args=tensor_args)

    obstacle_spheres = np.zeros((1, num_obst, 4))
    obstacle_spheres[0, :, :3] = np.random.uniform([0.6, -0.2, 0.6], [1., 0.2, 1.], (num_obst, 3))
    obstacle_spheres[0, :, 3] = np.random.uniform(0.1, 0.2, num_obst)
    obs = {'obstacle_spheres': torch.from_numpy(obstacle_spheres).to(**tensor_args)}

    opt_iters = 400
    torch.cuda.synchronize()
    t0 = time.time()
    for i in range(opt_iters + 1):
        trajectory_means, _, trajectories, _, costs, _ = planner.optimize(**obs)
    torch.cuda.synchronize()
    print(f'plan: {opt_iters + 1} optimize() calls in {(time.time() - t0) * 1e3:.1f} ms; mean cost {costs.mean().item():.4e}')

    # the final plan: the cheapest collision-free particle mean, checked at 8 states inside every interval as well as at the support
    # states (the planner's own GP interpolation), against the obstacle spheres
    best = planner.best_plans(n_interp=8, **obs)
    ee = ops.fk_link_positions(panda_fk, best.plan[-1:, :n_dof].contiguous())[0, -1]       # ee_link origin at t = T-1
    print('best plan: particle %d, collision-free %s, clearance to the spheres %.3f m, EE position error to the target %.4f m'
          % (best.particle.item(), bool(best.collision_free), best.clearance.item(), (ee - target_H[0, :3, 3]).norm().item()))
