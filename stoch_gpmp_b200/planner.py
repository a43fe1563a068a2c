"""StochGPMP with the reference's Python API, driving the sm_100a CUDA kernels.

  StochGPMP        drop-in for stoch_gpmp/planner.py:18-348 (one planning problem)
  StochGPMPBatch   the same loop over B independent problems at once (the reference has no problem
                   axis; B = 1 is exactly StochGPMP) — this is what shards over GPUs.

Host code only carries parameters and launches kernels through the C-ABI (ops.py / _lib.py):
  reset()      -> K1 sgpmp_prior_factor (init + sampling prior), K2 sgpmp_sample (initial means)
  optimize()   -> sgpmp_iterate (fused sample + cost + softmax + update, opt_iters per launch)
  sample_and_eval / _update_distribution / sample_trajectories -> K2 / K3 / K4
  optimize() with user-defined terms in cost_list             -> K2, K3 (+ the user's torch code), K4 per iteration
There is no CPU path: a CPU `tensor_args['device']` raises.

Differences from the reference that a user can observe (DESIGN.md §7):
  * eps comes from a counter-based Philox stream keyed by (seed, draw, problem, particle, sample), not
    from torch's global generator; runs are reproducible and independent of sharding.
  * the prior is factored once, in fp64, whatever `tensor_args['dtype']` is — fp32 planners that the
    reference cannot construct (README.md:33-35) work here.
  * samples are materialised lazily: the fused loop only writes the last iteration's samples when asked
    (`optimize(return_samples=...)`); `get_recent_samples()` regenerates them from the RNG counters.
"""
import collections
import time

import torch

from . import ops
from . import _lib


def print_info(iteration, max_iterations, start_time_iter, start_time, costs):
    """Same report line as stoch_gpmp/planner.py:668-672."""
    print(f'Iteration: {iteration:5}/{max_iterations:5} '
          f'| Iter Time: {time.time() - start_time_iter:.3f}'
          f'| Total Time: {time.time() - start_time:.3f} '
          f'| Cost: {costs.sum(-1).mean():.6f}')


PlanResult = collections.namedtuple('PlanResult', [
    'plan',                 # [B,T,d] the chosen particle mean, bit for bit
    'dense_plan',           # [B,P,d] its P = (T-1)(n_interp+1)+1 checked states; dense_plan[:, ::n_interp+1] == plan
    'dense_dt',             # time between two dense states: dt / (n_interp+1)
    'particle',             # [B] index of the chosen particle
    'cost',                 # [B] its ranking cost
    'collision_free',       # [B] bool: the chosen particle passed the check (no occupied map cell, clearance >= margin)
    'clearance',            # [B] its clearance to the obstacle spheres (+inf without a sphere field)
    'particle_costs',       # [B,NP] ranking cost of every particle mean
    'particle_clearance',   # [B,NP]
    'particle_hits',        # [B,NP] checked states in an occupied map cell
])


def prior_blocks(T, dt, sigma_start, sigma_gp, sigma_goal):
    """Per-DoF 2x2 blocks of the constant-velocity precision, host float64, expression order as in
    gp_factor.py:44-52 / mp_priors_multi.py:170-202.  Returns (D [T,3], O [T-1,4]) python lists."""
    qc = 1.0 / sigma_gp ** 2
    q11, q12, q22 = 12.0 * dt ** -3.0 * qc, -6.0 * dt ** -2.0 * qc, 4.0 * dt ** -1.0 * qc
    # Phi^T Q Phi with Phi = [[1, dt], [0, 1]]
    f11 = q11
    f12 = q11 * dt + q12
    f22 = (q11 * dt + q12) * dt + (q12 * dt + q22)
    ks = 1.0 / sigma_start ** 2
    D = []
    for t in range(T):
        d11 = d12 = d22 = 0.0
        if t >= 1:
            d11, d12, d22 = d11 + q11, d12 + q12, d22 + q22
        if t <= T - 2:
            d11, d12, d22 = d11 + f11, d12 + f12, d22 + f22
        if t == 0:
            d11, d22 = d11 + ks, d22 + ks
        if t == T - 1 and sigma_goal is not None:
            kg = 1.0 / sigma_goal ** 2
            d11, d22 = d11 + kg, d22 + kg
        D.append([d11, d12, d22])
    # O = -Q Phi
    O = [[-q11, -(q11 * dt + q12), -q12, -(q12 * dt + q22)] for _ in range(T - 1)]
    return D, O


class StochGPMPBatch:
    """StochGPMP over B independent planning problems.

    start_state [B, d]; multi_goal_states [B, G, d] (or None); `cost` a CostComposite whose CostGP /
    CostGoalPrior carry the same batched tensors; observation['obstacle_spheres'] [B, O, 4] or [1, O, 4].
    Tensors returned by optimize() have a leading B axis.  `problem_offset` is the global index of problem
    0 (RNG streams are keyed by global ids: sharding a batch over ranks does not change any result)."""

    _batched = True

    def __init__(self, num_particles_per_goal, num_samples, traj_len, opt_iters, dt=None, n_dof=None,
                 step_size=1., temperature=1., start_state=None, multi_goal_states=None,
                 initial_particle_means=None, cost=None,
                 sigma_start_init=None, sigma_start_sample=None, sigma_goal_init=None, sigma_goal_sample=None,
                 sigma_gp_init=None, sigma_gp_sample=None, seed=None, tensor_args=None,
                 problem_offset=0, **kwargs):
        if tensor_args is None:
            tensor_args = {'device': torch.device('cuda'), 'dtype': torch.float32}
        self.tensor_args = tensor_args
        dev = torch.device(tensor_args['device'])
        if dev.type != 'cuda':
            raise RuntimeError("stoch_gpmp_b200.StochGPMP needs a CUDA device (tensor_args['device']=%s); there is "
                               "no CPU fallback" % dev)
        _lib.load()                                   # fail loudly if the CUDA library is missing
        self.device, self.dtype = dev, tensor_args['dtype']
        # seed=None: the key is DRAWN from torch's global generator (ADVICE r1): unseeded planners / repeated trials get independent
        # noise as with the reference (which consumes the global generator), and torch.manual_seed() still makes a run reproducible
        self.seed = int(seed) if seed is not None else int(torch.randint(0, 2 ** 62, (1,)).item())
        self._draw = 0

        self.n_dof = n_dof
        self.d_state_opt = 2 * n_dof
        self.dt = dt
        self.traj_len = traj_len
        self.goal_directed = multi_goal_states is not None
        if self.goal_directed:
            assert multi_goal_states.dim() == (3 if self._batched else 2)
            self.num_goals = multi_goal_states.shape[-2]
        else:
            self.num_goals = 1
        self.num_particles_per_goal = num_particles_per_goal
        self.num_particles = num_particles_per_goal * self.num_goals
        self.num_samples = num_samples
        self.opt_iters = opt_iters
        self.step_size = step_size
        self.temperature = temperature
        self.sigma_start_init, self.sigma_start_sample = sigma_start_init, sigma_start_sample
        self.sigma_goal_init, self.sigma_goal_sample = sigma_goal_init, sigma_goal_sample
        self.sigma_gp_init, self.sigma_gp_sample = sigma_gp_init, sigma_gp_sample
        self.start_states = start_state
        self.multi_goal_states = multi_goal_states
        self.cost = cost
        self.problem_offset = int(problem_offset)
        if not _lib.load().sgpmp_dof_supported(n_dof):
            raise NotImplementedError("n_dof=%d is not instantiated in the CUDA library (csrc/sgpmp_dof_list.inc)" % n_dof)

        self._weights_raw = None
        self._last = None
        self.reset(start_state, multi_goal_states, initial_particle_means=initial_particle_means)

    # ------------------------------------------------------------------------------------------------
    def _b(self, t, inner_dims):
        """Bring a user tensor to [B, ...inner] on the planner's device/dtype."""
        t = torch.as_tensor(t).detach().to(device=self.device, dtype=self.dtype)
        if t.dim() == inner_dims:
            t = t.unsqueeze(0)
        return t.contiguous()

    def _shape(self, S=None, G=None, K=None):
        if S is None and G is None and K is None:
            if getattr(self, "_shape_cache", None) is None:
                self._shape_cache = ops.make_shape(self.num_problems, self.num_goals, self.num_particles_per_goal, self.num_samples,
                                                   self.traj_len, self.n_dof, self.dtype, self.problem_offset)
            return self._shape_cache
        return ops.make_shape(self.num_problems, self.num_goals if G is None else G,
                              self.num_particles_per_goal if K is None else K,
                              self.num_samples if S is None else S, self.traj_len, self.n_dof, self.dtype,
                              self.problem_offset)

    def _factor(self, sigma_start, sigma_gp, sigma_goal, which):
        D, O = prior_blocks(self.traj_len, self.dt, sigma_start, sigma_gp, sigma_goal if self.goal_directed else None)
        Dt = torch.tensor([D], dtype=torch.float64, device=self.device)
        Ot = torch.tensor([O], dtype=torch.float64, device=self.device)
        tables, not_pd = ops.prior_factor(Dt, Ot)
        bad = int(not_pd[0].item())
        if bad:
            # reference: ValueError from torch's PositiveDefinite constraint (mp_priors_multi.py:106)
            raise ValueError("%s prior precision is not positive definite in fp64 (pivot block t=%d): check "
                             "sigma_start/sigma_gp/sigma_goal (%g, %g, %s) and dt=%g"
                             % (which, bad - 1, sigma_start, sigma_gp, sigma_goal, self.dt))
        return tables[0].contiguous(), (Dt[0], Ot[0])

    def const_vel_trajectories(self, start_state, multi_goal_states):
        """'const_vel' initial means [G,K,T,d] (+ leading B for the batch class); planner.py:142-155."""
        return self._out(self._const_vel(start_state, multi_goal_states))

    def _const_vel(self, start_state, multi_goal_states):
        """[B,G,K,T,d]; velocity = (goal-start)/(T*dt) (planner.py:149), unlike the INIT prior's mean."""
        n, T, K = self.n_dof, self.traj_len, self.num_particles_per_goal
        s = self._b(start_state, 1)[:, None, :n]                                  # [B,1,n]
        g = self._b(multi_goal_states, 2)[:, :, :n]                               # [B,G,n]
        i = torch.arange(T, device=self.device, dtype=self.dtype).view(1, 1, T, 1)
        pos = s.unsqueeze(2) * (T - i - 1) / (T - 1) + g.unsqueeze(2) * i / (T - 1)       # [B,G,T,n]
        vel = ((g - s) / (T * self.dt)).unsqueeze(2).expand(-1, -1, T, -1)
        traj = torch.cat([pos, vel], dim=-1)                                      # [B,G,T,d]
        return traj.unsqueeze(2).expand(-1, -1, K, -1, -1).contiguous()

    def _init_prior_means(self):
        """Straight-line means of the INIT prior [B,G,T,d] (mp_priors_multi.py:130-168; /((T-1)*dt))."""
        n, T = self.n_dof, self.traj_len
        s = self.start_state
        if not self.goal_directed:
            return s[:, None, None, :].expand(-1, 1, T, -1).contiguous()
        g = self.multi_goal_states
        ns = T - 1
        i = torch.arange(T, device=self.device, dtype=self.dtype).view(1, 1, T, 1)
        pos = s[:, None, None, :n] * (ns - i) * 1. / ns + g[:, :, None, :n] * i * 1. / ns
        vel = ((g[:, :, :n] - s[:, None, :n]) / (ns * self.dt)).unsqueeze(2).expand(-1, -1, T, -1)
        return torch.cat([pos, vel], dim=-1).contiguous()

    def reset(self, start_state=None, multi_goal_states=None, initial_particle_means=None, _init_eps=None):
        """(Re)build priors and particle means (planner.py:181-227)."""
        if start_state is not None:
            self.start_state = self._b(start_state, 1)
        if multi_goal_states is not None:
            self.multi_goal_states = self._b(multi_goal_states, 2)
        self.num_problems = self.start_state.shape[0]
        B, G, K, T, d = self.num_problems, self.num_goals, self.num_particles_per_goal, self.traj_len, self.d_state_opt

        if initial_particle_means is not None:
            if isinstance(initial_particle_means, str):
                if initial_particle_means != 'const_vel':
                    raise ValueError("unknown initial_particle_means mode %r" % initial_particle_means)
                pm = self._const_vel(self.start_state, self.multi_goal_states)
            else:
                pm = self._b(initial_particle_means, 4)
                if tuple(pm.shape) != (B, G, K, T, d):
                    raise AssertionError("initial_particle_means must be [G,K,T,d]" + (" with a leading B" if self._batched else ""))
        else:
            tab_init, _ = self._factor(self.sigma_start_init, self.sigma_gp_init, self.sigma_goal_init, "initialisation")
            mu0 = self._init_prior_means()                                        # [B,G,T,d]
            sh = self._shape(S=K, G=G, K=1)
            eps = None
            if _init_eps is not None:   # parity hook: reference draw layout [K, G, M] per problem -> [B,G,T,d,K]
                eps = self._b(_init_eps, 3).reshape(B, K, G, T, d).permute(0, 2, 3, 4, 1).contiguous()
            x = ops.sample(sh, tab_init, mu0, eps_in=eps, seed=self.seed, draw=self._draw)    # [B,G,T,d,K]
            self._draw += 1
            pm = x.permute(0, 1, 4, 2, 3).contiguous()                            # [B,G,K,T,d]
        self._means = pm.reshape(B, G * K, T, d).contiguous().clone()

        self._tables, (self._D, self._O) = self._factor(self.sigma_start_sample, self.sigma_gp_sample,
                                                        self.sigma_goal_sample, "sampling")
        self._lowered = self.cost.lower(B, G, self.device, self.dtype) if self.cost is not None else None
        # the reference draws (and keeps) one sample batch here (planner.py:227); we only reserve its draw
        # index and materialise it if `state_samples` is read.
        self._state_samples_src = (self._means.clone(), self._draw, self.num_samples)
        self._state_samples = None
        self._draw += 1
        self._Sigma_inv = None
        self._last = None
        self._shape_cache = None
        import os
        self._lowlat_env = os.environ.get("SGPMP_LOWLAT")      # read once per reset(): optimize() is host-bound for one problem
        self._warm_kernels()

    _warm = True        # GPMPBatch (another algorithm on the same state) switches the warm-up off

    def _warm_kernels(self):
        """The first launch of a kernel loads its code (CUDA loads functions lazily; 5 ms for the fused kernel, 40 ms for the three
        kernels of the low-latency form).  The reference's scripts time their optimize() loop from the first call, so that load
        is taken here, at construction: one iteration of the form optimize() will pick, on a scratch copy of the means, with a
        far-away placeholder sphere when the cost list has a sphere field (same kernel family; the sphere count is a run-time
        loop).  No state of the planner changes.  $SGPMP_WARMUP=0 skips it."""
        import os
        if (not self._warm or self._lowered is None or self._lowered.custom or os.environ.get("SGPMP_WARMUP") == "0" or
                self.num_problems * self.num_particles > 4096):
            return
        try:
            obs = None
            if self._lowered.sphere_sigma is not None:
                obs = torch.tensor([[[1e3, 1e3, 1e3, 1.0]]], dtype=self.dtype, device=self.device)
            desc = self._lowered.desc(self.temperature, obs)
            forms = {self._lowlat(1), self._lowlat(self.opt_iters), self._lowlat(1 << 20)}     # single call, default, long plan
            for ll in forms:
                ops.iterate(self._shape(), desc, self._tables, self.step_size, 1, self._means.clone(), seed=self.seed, draw0=self._draw,
                            want_samples=False, lowlat=ll)
        except NotImplementedError:
            pass        # un-lowerable shape: optimize() itself will raise with the reason
        finally:
            self._lowered._spheres_src = None          # the next real call patches the descriptor with the caller's spheres
            if self._lowered.sphere_sigma is not None:
                self._lowered.desc(self.temperature, None)

    # ---- attributes users read -------------------------------------------------------------------------
    def _out(self, t):
        return t

    @property
    def _weights(self):
        """Softmax weights of the last iteration as the reference keeps them, [NP, S, 1, 1] (planner.py:264-266).  Built on
        access: every tensor view costs the host ~1.2 us, and optimize() is host-bound when it is called once per iteration."""
        w = self._weights_raw
        if w is None:
            return None
        w = self._out(w)
        return w.reshape(*w.shape, 1, 1)

    @property
    def particle_means(self):
        return self._out(self._means)

    @particle_means.setter
    def particle_means(self, v):
        self._means = self._b(v, 3).reshape(self._means.shape).contiguous().clone()

    def _materialise(self, src):
        means, draw, S = src
        x = ops.sample(self._shape(S=S), self._tables, means, seed=self.seed, draw=draw)
        return x.permute(0, 1, 4, 2, 3)                   # view [B,NP,S,T,d] of the S-minor buffer

    @property
    def state_samples(self):
        if self._state_samples is None:
            if self._state_samples_src is None:       # the last optimize() wrote its samples: view of the S-minor buffer
                self._state_samples = self._samples_sminor.permute(0, 1, 4, 2, 3)
            else:
                self._state_samples = self._materialise(self._state_samples_src)
        return self._out(self._state_samples)

    @property
    def Sigma_inv(self):
        """Dense [M,M] precision (planner.py:226) assembled on demand from the 2x2 blocks."""
        if self._Sigma_inv is None:
            n, T, d = self.n_dof, self.traj_len, self.d_state_opt
            eye = torch.eye(n, dtype=torch.float64, device=self.device)
            P = torch.zeros(T * d, T * d, dtype=torch.float64, device=self.device)
            Dm, Om = self._D, self._O
            for t in range(T):
                Db = torch.stack([torch.stack([Dm[t, 0], Dm[t, 1]]), torch.stack([Dm[t, 1], Dm[t, 2]])])
                P[t * d:(t + 1) * d, t * d:(t + 1) * d] = torch.kron(Db, eye)
                if t + 1 < T:
                    Ob = torch.kron(Om[t].reshape(2, 2), eye)
                    P[(t + 1) * d:(t + 2) * d, t * d:(t + 1) * d] = Ob
                    P[t * d:(t + 1) * d, (t + 1) * d:(t + 2) * d] = Ob.T
            self._Sigma_inv = P.to(self.dtype)
        return self._Sigma_inv

    # ---- separate-kernel path (reference method names) ------------------------------------------------
    def _desc(self, observation):
        if self._lowered is None:
            raise NotImplementedError("StochGPMP needs a CostComposite (cost=...)")
        if self._lowered.goal_K is not None and (self._lowered.goal_K != self.num_particles_per_goal or
                                                 self._lowered.goal_S != self.num_samples):
            # the reference fails in CostGoalPrior's reshape (cost_functions.py:379) on this mismatch
            raise RuntimeError("CostGoalPrior was built with num_particles_per_goal=%s, num_samples=%s but the planner "
                               "uses %d, %d" % (self._lowered.goal_K, self._lowered.goal_S,
                                                self.num_particles_per_goal, self.num_samples))
        return self._lowered.desc(self.temperature, observation.get('obstacle_spheres', None))

    def sample_and_eval(self, _eps=None, **observation):
        """planner.py:239-261: (vel samples, pos samples, vel means, pos means, costs)."""
        n = self.n_dof
        sh = self._shape()
        xs = ops.sample(sh, self._tables, self._means, eps_in=_eps, seed=self.seed, draw=self._draw)
        self._draw += 1
        self._samples_sminor = xs
        self._state_samples = xs.permute(0, 1, 4, 2, 3)
        costs = ops.cost(sh, self._desc(observation), self._tables, xs, self._means)
        if self._lowered.custom:
            costs = costs + self._custom_costs(xs, observation)
        ss = self._state_samples
        return (self._out(ss[..., -n:]), self._out(ss[..., :n]),
                self._out(self._means[..., -n:].clone()), self._out(self._means[..., :n].clone()), self._out(costs))

    def _custom_costs(self, xs, observation):
        """User-defined terms of cost_list (objects the kernels cannot lower), evaluated by the user's torch code on the
        materialised samples xs [B,NP,T,d,S] with the reference's calling convention (cost_functions.py:47-56) -> [B,NP,S]."""
        B, NP, T, d, S = xs.shape
        trajs = xs.permute(0, 1, 4, 2, 3).reshape(B * NP * S, T, d)
        c = self._lowered.custom_costs(trajs, **observation)
        return torch.as_tensor(c, device=self.device).to(self.dtype).reshape(B, NP, S)

    def _optimize_separate(self, opt_iters, observation, _eps=None):
        """optimize() for cost lists with user-defined terms: the reference-method iteration K2 sample -> K3 cost (+ IS) -> user
        terms (torch) -> K4 update, with the samples materialised every iteration (the fused kernel never materialises them, so it
        cannot hand them to Python code).  Same RNG stream and same outputs as ops.iterate()."""
        sh = self._shape()
        desc = self._desc(observation)
        out = None
        for it in range(opt_iters):
            eps = None if _eps is None else _eps[it].contiguous()
            xs = ops.sample(sh, self._tables, self._means, eps_in=eps, seed=self.seed, draw=self._draw)
            self._draw += 1
            costs = ops.cost(sh, desc, self._tables, xs, self._means) + self._custom_costs(xs, observation)
            means_pre = self._means.clone()
            grad, w = ops.update(sh, self.temperature, self.step_size, costs.contiguous(), xs, self._means)
            out = dict(means_pre=means_pre, samples=xs, costs=costs, weights=w, grad=grad)
        return out

    def _update_distribution(self, costs, traj_samples=None):
        """planner.py:263-275.  `traj_samples` must be the samples of the last sample_and_eval()."""
        costs = costs.reshape(self.num_problems, self.num_particles, self.num_samples).contiguous()
        grad, w = ops.update(self._shape(), self.temperature, self.step_size, costs, self._samples_sminor, self._means)
        self._weights_raw = w
        return self._out(grad)

    def _lowlat(self, n_iters):
        """Few problems (the reference's own use: ONE): the fused kernel's thread-per-sample mapping would leave the GPU idle, so
        optimize() runs the low-latency form (three short launches per iteration, csrc/sgpmp_lowlat.cu).  $SGPMP_LOWLAT=0/1
        overrides the choice."""
        env = self._lowlat_env
        if env is not None:
            return env != "0"
        # measured on B200, us per iteration, fused (cluster) form -> low-latency form: one Panda problem 89.9 -> 31.2, one planar
        # problem 33.3 -> 25.1.  A call that runs a SINGLE cheap (no link fields) iteration is host-bound either way and the fused
        # form costs the host one launch instead of three (planar example, 501 single-iteration calls: 100 against 142 ms).
        small = self.num_problems * self.num_particles * self.num_samples <= 148 * 64
        heavy = self._lowered is not None and self._lowered.fk is not None
        return small and (heavy or n_iters >= 4)

    # ---- the hot loop ------------------------------------------------------------------------------------
    def optimize(self, opt_iters=None, debug=False, return_samples=None, _eps=None, **observation):
        """planner.py:277-317.  Runs `opt_iters` iterations in one fused launch and returns the reference's
        6-tuple for the LAST iteration: (pos means BEFORE the update, vel means BEFORE the update,
        pos samples, vel samples, costs [NP,S], grad [NP,T,d]).  With return_samples=False the two sample
        entries are None (nothing is written to HBM); get_recent_samples() can still rebuild them."""
        if opt_iters is None:
            opt_iters = self.opt_iters
        if return_samples is None:
            return_samples = not self._batched
        n = self.n_dof
        desc = self._desc(observation)
        sh = self._shape()
        start_time = time.time()
        chunks = [opt_iters]
        if debug:           # report every 50 iterations like planner.py:301-302
            chunks = [1] + [min(50, opt_iters - 1 - k) for k in range(0, max(opt_iters - 1, 0), 50)]
        done = 0
        out = None
        for ci, c in enumerate(chunks):
            if c <= 0:
                continue
            t_iter = time.time()
            eps = None if _eps is None else _eps[done:done + c].contiguous()
            last_chunk = (done + c == opt_iters)
            if self._lowered.custom:
                out = self._optimize_separate(c, observation, _eps=eps)
                if not (return_samples and last_chunk):
                    out['samples'] = None
            else:
                out = ops.iterate(sh, desc, self._tables, self.step_size, c, self._means, eps_in=eps, seed=self.seed,
                                  draw0=self._draw, want_samples=bool(return_samples and last_chunk), lowlat=self._lowlat(c),
                                  validate=eps is not None)
                self._draw += c
            done += c
            if debug:
                print_info(done - 1, opt_iters, t_iter, start_time, out['costs'])
        self._last = dict(means_pre=out['means_pre'], draw=self._draw - 1, eps=None if _eps is None else _eps[-1],
                          samples=out['samples'])
        self._weights_raw = out['weights']
        pos_s = vel_s = None
        if out['samples'] is not None:
            # views are built from the per-problem tensor when there is no batch axis to return: every view costs the host ~1.2 us
            # and this call is host-bound in the reference's usage (one optimize() per iteration); `state_samples` builds its
            # [B,NP,S,T,d] view on access
            xs = out['samples']
            ss = xs.permute(0, 1, 4, 2, 3) if self._batched else xs[0].permute(0, 3, 1, 2)
            self._samples_sminor = xs
            self._state_samples = None
            self._state_samples_src = None
            pos_s, vel_s = ss[..., :n], ss[..., -n:]
        elif _eps is None:
            # nothing was written: `state_samples` (and _get_traj) regenerate THIS iteration's samples lazily from the RNG
            # counters, so that they always pair with the weights of the same iteration (ADVICE r1)
            self._state_samples = None
            self._state_samples_src = (out['means_pre'], self._draw - 1, self.num_samples)
        mp = self._out(out['means_pre'])
        return (mp[..., :n], mp[..., -n:], pos_s, vel_s, self._out(out['costs']), self._out(out['grad']))

    def optimize_split(self, opt_iters=None, group=None, return_samples=False, **observation):
        """Split-particle mode (SURVEY §8e): the S samples of every particle are divided over the ranks of `group`;
        this rank draws and scores samples [rank*S/R, (rank+1)*S/R) (RNG streams are keyed by GLOBAL sample index,
        so the union over ranks is exactly the single-GPU sample set).  Per iteration: one fused launch (sample -> cost ->
        local softmax statistics, nothing materialised), ONE ncclAllGather of the per-particle (m, Z, A) blocks issued from C
        on the compute stream, one launch that merges them by log-sum-exp and applies the update identically on every rank.
        All iterations are enqueued by one call (ops.iterate_split_particles); the arithmetic split is planner.py:263-275.
        Returns (pos means before the last update, vel means, local pos samples, local vel samples, local costs, grad);
        the two sample entries are None unless return_samples (they are then regenerated from the RNG counters)."""
        import torch.distributed as dist
        from . import parallel
        if opt_iters is None:
            opt_iters = self.opt_iters
        if dist.is_available() and dist.is_initialized():
            world, rank = dist.get_world_size(group), dist.get_rank(group)
        else:
            world, rank = 1, 0
        if self.num_samples % world:
            raise ValueError("num_samples=%d is not divisible by the %d ranks of the group" % (self.num_samples, world))
        s_loc = self.num_samples // world
        n = self.n_dof
        desc = self._desc(observation)
        if self._lowered.custom:
            raise NotImplementedError("split-particle mode runs the fused statistics kernel; user-defined cost objects need the "
                                      "separate-kernel iteration of optimize()")
        sh_loc = ops.make_shape(self.num_problems, self.num_goals, self.num_particles_per_goal, s_loc, self.traj_len, n,
                                self.dtype, self.problem_offset, sample_gid0=rank * s_loc)
        comm = parallel.NcclComm.for_group(group, self.device).handle if world > 1 else None
        out = ops.iterate_split_particles(sh_loc, desc, self._tables, self.step_size, opt_iters, self._means, self.seed, self._draw,
                                          comm=comm, n_ranks=world)
        self._draw += opt_iters
        self._split_keepalive = out["_keepalive"]
        pos_s = vel_s = None
        if return_samples:
            xs = ops.sample(sh_loc, self._tables, out["means_pre"], seed=self.seed, draw=self._draw - 1)
            ss = xs.permute(0, 1, 4, 2, 3)
            pos_s, vel_s = self._out(ss[..., :n]), self._out(ss[..., -n:])
        mp = out["means_pre"]
        return (self._out(mp[..., :n]), self._out(mp[..., -n:]), pos_s, vel_s, self._out(out["costs"]), self._out(out["grad"]))

    def get_recent_samples(self):
        """planner.py:330-337: (position samples, velocity samples) of the last iteration, fresh tensors."""
        if self._last is None:
            raise AttributeError("optimize() has not been called yet")
        n = self.n_dof
        if self._last['samples'] is not None:
            ss = self._last['samples'].permute(0, 1, 4, 2, 3)
        else:
            xs = ops.sample(self._shape(), self._tables, self._last['means_pre'], eps_in=self._last['eps'],
                            seed=self.seed, draw=self._last['draw'])
            ss = xs.permute(0, 1, 4, 2, 3)
        return self._out(ss[..., :n]).detach().clone(), self._out(ss[..., -n:]).detach().clone()

    def weighted_covariance(self, tensor_cores=True):
        """Diagnostic with no reference counterpart (the reference keeps Sigma^-1 fixed, planner.py:226): the weighted sample
        covariance  sum_s w_s (x_s - mu)(x_s - mu)^T  [NP, M, M] of the LAST optimize() iteration, with the weights and the
        pre-update means of that iteration.  fp32: tcgen05 tensor-core kernel (csrc/sgpmp_cov.cu)."""
        if self._last is None:
            raise AttributeError("optimize() has not been called yet")
        xs = self._last['samples']
        if xs is None:
            xs = ops.sample(self._shape(), self._tables, self._last['means_pre'], eps_in=self._last['eps'], seed=self.seed,
                            draw=self._last['draw'])
        return self._out(ops.weighted_cov(self._shape(), xs, self._last['means_pre'], self._weights_raw.contiguous(), tensor_cores))

    def sample_trajectories(self, num_samples_per_particle):
        """planner.py:339-348."""
        n = self.n_dof
        xs = ops.sample(self._shape(S=num_samples_per_particle), self._tables, self._means, seed=self.seed, draw=self._draw)
        self._draw += 1
        self._state_samples = xs.permute(0, 1, 4, 2, 3)
        return self._out(self._state_samples[..., :n]), self._out(self._state_samples[..., -n:])

    def _get_traj(self, mode='best'):
        if mode == 'best':
            ind = self._weights.argmax()
            return self.state_samples.reshape(-1, self.num_samples, self.traj_len, self.d_state_opt)[ind].clone()
        raise ValueError('Unidentified sampling mode in get_next_action')

    def best_plans(self, n_interp=8, margin=0.0, **observation):
        """The final step of planning: one plan per problem, with a yes/no answer on whether it is collision-free.  No reference
        counterpart (DESIGN.md §7).  Returns a PlanResult (fields above; StochGPMP drops the B axis).

        Works on the CURRENT particle means (`particle_means`, i.e. after the last update), not on the pre-update means that
        optimize() returns.  Every mean is checked at its support states t >= 1 and at n_interp states inside every interval: the
        constant-velocity GP prior's own interpolation (cubic Hermite in (q, qdot)), so the check holds for the trajectory model the
        planner optimises, not only at its support states.  The obstacle spheres of `observation` (as optimize() takes them) are
        checked geometrically: clearance is the least |p - c| - r over the sphere field's points (link-frame origins and its link
        interpolation) and spheres, whatever the field type.  Occupancy maps of the cost are checked cell by cell.  The
        self-collision field is NOT checked: its RBF over all link pairs, adjacent links included, defines no distance to hold
        against a margin.

        A particle is collision-free when no checked state lies in an occupied map cell and its clearance is >= margin (in
        metres).  The plan of a problem is its cheapest collision-free particle (ties to the lowest index); with none, the
        cheapest particle overall (NaN costs last), with collision_free False.  The ranking cost is CostComposite.eval of the
        mean without the importance-sampling term."""
        low = self._lowered
        if low is None:
            raise NotImplementedError("best_plans needs a CostComposite (cost=...)")
        if low.custom:
            raise NotImplementedError("best_plans ranks the means with the CUDA cost kernel; user-defined cost objects (%s) are not "
                                      "supported" % ", ".join(type(c).__name__ for c in low.custom))
        B, NP = self.num_problems, self.num_particles
        sh = self._shape(S=1)
        desc = low.desc(0.0, observation.get('obstacle_spheres', None))
        # [B,NP,T,d] is the S-minor sample layout [B,NP,T,d,1]; means=None drops the IS term; the goal of particle p is p // K
        costs = ops.cost(sh, desc, None, self._means.unsqueeze(-1), None).reshape(B, NP)
        r = ops.select_plans(sh, desc, self._means, costs, n_interp, margin)
        particle = r['particle'].long()
        pick = particle.unsqueeze(1)
        o = self._out
        return PlanResult(plan=o(r['plan']), dense_plan=o(r['dense']), dense_dt=self.dt / (n_interp + 1), particle=o(particle),
                          cost=o(costs.gather(1, pick).squeeze(1)), collision_free=o(r['ok'].bool()),
                          clearance=o(r['clearance'].gather(1, pick).squeeze(1)), particle_costs=o(costs),
                          particle_clearance=o(r['clearance']), particle_hits=o(r['hits']))


class StochGPMP(StochGPMPBatch):
    """Single-problem planner with exactly the reference's shapes (no leading B axis)."""

    _batched = False

    def _out(self, t):
        return None if t is None else t[0]

    def reset(self, start_state=None, multi_goal_states=None, initial_particle_means=None, _init_eps=None):
        if initial_particle_means is not None and not isinstance(initial_particle_means, str):
            initial_particle_means = torch.as_tensor(initial_particle_means).unsqueeze(0)
        if start_state is not None:
            start_state = torch.as_tensor(start_state).reshape(1, -1)
        if multi_goal_states is not None:
            multi_goal_states = torch.as_tensor(multi_goal_states).unsqueeze(0)
        return super().reset(start_state, multi_goal_states, initial_particle_means, _init_eps=_init_eps)

    def sample_and_eval(self, _eps=None, **observation):
        return super().sample_and_eval(_eps=None if _eps is None else _eps.unsqueeze(0), **observation)

    def optimize(self, opt_iters=None, debug=False, return_samples=None, _eps=None, **observation):
        if _eps is not None:
            _eps = _eps.unsqueeze(1)             # [n_iters, 1, NP, T, d, S]
        return super().optimize(opt_iters, debug, return_samples, _eps, **observation)


def __getattr__(name):
    # `from stoch_gpmp.planner import GPMP` (planner.py:352) keeps working: the Gauss-Newton planner lives in gpmp.py
    if name in ('GPMP', 'GPMPBatch'):
        from . import gpmp
        return getattr(gpmp, name)
    raise AttributeError("module %r has no attribute %r" % (__name__, name))
