"""GPU parity tests, kernel by kernel, through the C-ABI (stoch_gpmp_b200.ops -> libsgpmp.so).

Checker = oracle/ (numpy) and the golden vectors produced by the real reference (tests/golden).
Tolerances: fp64 1e-10 relative (factor-dependent quantities are conditioning-limited on one case, see
helpers.FACTOR_TOL_F64), fp32 1e-5 relative against the reference run with the same prior factor.
"""
import numpy as np
import pytest
import torch

from oracle import philox as OPH
from oracle import planner as OP
from oracle import prior as P
from oracle import sampler as SMP
from oracle import fk as OFK

from helpers import (GOLDEN_C3, eps_from_rng_state, GOLDEN, GOLDEN_F32, GOLDEN_F64, FACTOR_TOL_F64, TOL_F32, TOL_F64, eps_ref_to_traj, from_sminor,
                     load, n_iters, rel, to_sminor)

pytestmark = pytest.mark.gpu


def _ops():
    from stoch_gpmp_b200 import ops
    return ops


def _tables(spec, dev, which='sample'):
    from stoch_gpmp_b200.planner import prior_blocks
    goal = spec[f'sigma_goal_{which}'] if spec.get('goals') is not None else None
    D, O = prior_blocks(spec['T'], spec['dt'], spec[f'sigma_start_{which}'], spec[f'sigma_gp_{which}'], goal)
    Dt = torch.tensor([D], dtype=torch.float64, device=dev)
    Ot = torch.tensor([O], dtype=torch.float64, device=dev)
    tables, bad = _ops().prior_factor(Dt, Ot)
    assert int(bad[0]) == 0
    return tables[0].contiguous()


def _lowered(spec, dev, dtype, B=1):
    """Build product cost objects from a spec and lower them."""
    from stoch_gpmp_b200.costs.cost_functions import CostCollision, CostComposite, CostGP, CostGoalPrior
    from stoch_gpmp_b200.costs.fields import LinkDistanceField
    from stoch_gpmp_b200.envs.occupancy import ObstacleMap
    from stoch_gpmp_b200.robots import PandaFK
    ta = dict(device=dev, dtype=dtype)
    n, T = spec['n_dof'], spec['T']
    if spec.get('cost_sigma_start') is None:
        from stoch_gpmp_b200.costs.cost_functions import CostGPTrajectory
        cl = [CostGPTrajectory(n, T, torch.tensor(spec['start'], **ta), spec['dt'], dict(sigma_gp=spec['cost_sigma_gp']), ta)]
    else:
        cl = [CostGP(n, T, torch.tensor(spec['start'], **ta), spec['dt'],
                     dict(sigma_start=spec['cost_sigma_start'], sigma_gp=spec['cost_sigma_gp']), ta)]
    if spec.get('goals') is not None and spec.get('sigma_goal_prior') is not None:
        cl.append(CostGoalPrior(n, T, multi_goal_states=torch.tensor(spec['goals'], **ta), num_particles_per_goal=spec['K'],
                                num_samples=spec['S'], sigma_goal_prior=spec['sigma_goal_prior'], tensor_args=ta))
    FK = None
    if spec.get('self_margin') is not None:
        from stoch_gpmp_b200.costs.fields import LinkSelfDistanceField
        FK = PandaFK()
        ikw = {}
        if spec.get('self_num_interpolate'):
            ikw = dict(num_interpolate=spec['self_num_interpolate'], link_interpolate_range=list(spec['self_interp_range']))
        cl.append(CostCollision(n, T, field=LinkSelfDistanceField(margin=spec['self_margin'], tensor_args=ta, **ikw), sigma_coll=spec['sigma_self']))
    if 'map' in spec:
        H = spec['map'].shape[0]
        om = ObstacleMap([2, 2], 1.0, tensor_args=ta)
        om.map = spec['map'].copy()
        om.cell_size = spec['map_cell_size']
        om.origin_xi, om.origin_yi = spec['map_origin']
        cl.append(CostCollision(n, T, field=om, sigma_coll=spec['sigma_coll']))
    if 'spheres' in spec:
        FK = PandaFK()
        ikw = {}
        if spec.get('num_interpolate'):
            ikw = dict(num_interpolate=spec['num_interpolate'], link_interpolate_range=list(spec['interp_range']))
        cl.append(CostCollision(n, T, field=LinkDistanceField(field_type=spec.get('field_type', 'rbf'), clamp_sdf=spec.get('clamp_sdf', False),
                                                              tensor_args=ta, **ikw), sigma_coll=spec['sigma_coll']))
    if spec.get('ee_target') is not None:
        from stoch_gpmp_b200.costs.cost_functions import CostGoal
        from stoch_gpmp_b200.costs.fields import EESE3DistanceField
        FK = PandaFK()
        fld = EESE3DistanceField(torch.tensor(spec['ee_target'], **ta).reshape(1, 4, 4), w_pos=spec['ee_w_pos'], w_rot=spec['ee_w_rot'],
                                 square=spec['ee_square'], tensor_args=ta)
        cl.append(CostGoal(n, T, field=fld, sigma_goal=spec['sigma_ee_goal'], tensor_args=ta))
    comp = CostComposite(n, T, cl, FK=FK, tensor_args=ta)
    G = spec['G']
    return comp, comp.lower(B, G, dev, dtype)


def _obs(spec, dev, dtype):
    return {'obstacle_spheres': torch.tensor(spec['spheres'], device=dev, dtype=dtype).unsqueeze(0)} if 'spheres' in spec else {}


# --------------------------------------------------------------------------------------------- K1 prior
@pytest.mark.parametrize("name", GOLDEN)
def test_prior_tables_match_oracle(name, cuda):
    spec = OP.spec_from_golden(load(name))
    tab = _tables(spec, cuda).cpu().numpy()
    D, O, fac = OP.sampling_prior(spec)
    G = np.stack([tab[:, 0], tab[:, 1], tab[:, 2]], 1)
    Go = np.stack([fac['G'][:, 0, 0], fac['G'][:, 1, 0], fac['G'][:, 1, 1]], 1)
    Ho = fac['H'].reshape(-1, 4)
    # same operation order, IEEE double, no FMA: expected bit-identical; allow a few ulp
    assert rel(G, Go) < 1e-14
    assert rel(tab[:, 3:7], Ho) < 1e-14
    assert np.array_equal(tab[:, 7:10], np.stack([D[:, 0, 0], D[:, 0, 1], D[:, 1, 1]], 1))
    assert np.array_equal(tab[:-1, 10:14], O.reshape(-1, 4))


@pytest.mark.parametrize("name", GOLDEN_F64)
def test_prior_dense_L_matches_reference(name, cuda):
    g = load(name)
    spec = OP.spec_from_golden(g)
    L = _ops().prior_dense_L(_tables(spec, cuda), spec['n_dof'], torch.float64).cpu().numpy()
    assert rel(L, g['L']) < FACTOR_TOL_F64.get(name, TOL_F64)


@pytest.mark.parametrize("T,n", [(64, 2), (128, 4), (256, 7), (1024, 14)])
def test_prior_sweep_fp64(T, n, cuda):
    """C5: prior construction for long horizons; moments against the per-DoF dense covariance
    (valid because the precision decouples per DoF, SURVEY §8a-2)."""
    spec = dict(T=T, dt=0.02, goals=np.zeros((1, 2 * n)), sigma_start_sample=1e-3, sigma_gp_sample=3.0, sigma_goal_sample=1e-3)
    tab = _tables(spec, cuda)
    D, O = P.precision_blocks(T, 0.02, 1e-3, 3.0, 1e-3)
    fac = P.banded_factor(D, O)
    t = tab.cpu().numpy()
    assert rel(t[:, [0, 1, 2]], np.stack([fac['G'][:, 0, 0], fac['G'][:, 1, 0], fac['G'][:, 1, 1]], 1)) < 1e-13
    if T <= 256:
        L1 = _ops().prior_dense_L(tab, 1, torch.float64).cpu().numpy()        # one DoF: 2T x 2T
        Sigma = np.linalg.inv(P.dense_from_blocks(D, O, 1))
        assert rel(L1 @ L1.T, Sigma) < 1e-5
    if T * n <= 512:
        Ln = _ops().prior_dense_L(tab, n, torch.float64).cpu().numpy()
        assert rel(Ln, P.dense_scale_tril(fac['G'], fac['H'], n)) < 1e-12


def test_prior_not_pd_flag(cuda):
    D, O = P.precision_blocks(8, 0.1, 1.0, 1.0, 1.0)
    D[3] *= -1
    Dt = torch.tensor(np.stack([D[:, 0, 0], D[:, 0, 1], D[:, 1, 1]], 1)[None], device=cuda)
    Ot = torch.tensor(O.reshape(1, -1, 4), device=cuda)
    _, bad = _ops().prior_factor(Dt.contiguous(), Ot.contiguous())
    assert int(bad[0]) == 1 + 3


# -------------------------------------------------------------------------------------------- K2 sample
@pytest.mark.parametrize("name", GOLDEN)
def test_sample_injected_eps_matches_reference(name, cuda):
    g = load(name)
    spec = OP.spec_from_golden(g)
    f32 = spec['dtype'] == 'float32'
    dt = torch.float32 if f32 else torch.float64
    pre0 = 'sameL_' if f32 else ''
    T, d = spec['T'], 2 * spec['n_dof']
    tab = _tables(spec, cuda)
    sh = _ops().make_shape(1, spec['G'], spec['K'], spec['S'], T, spec['n_dof'], dt)
    for it in range(n_iters(g, pre0)):
        pre = f'{pre0}it{it}_'
        eps = torch.tensor(to_sminor(eps_ref_to_traj(g[pre + 'eps'], T, d)), device=cuda)
        mu = torch.tensor(g[pre + 'means_pre'][None], device=cuda)
        x = from_sminor(_ops().sample(sh, tab, mu, eps_in=eps).cpu().numpy())[0]
        tol = TOL_F32 if f32 else FACTOR_TOL_F64.get(name, TOL_F64)
        assert rel(x, g[pre + 'samples']) < tol


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("T,n,S", [(16, 2, 40), (7, 3, 33), (64, 7, 64)])
def test_sample_inkernel_rng_matches_oracle_stream(dtype, T, n, S, cuda):
    """The kernel's Philox/Box-Muller stream == oracle/philox.py (odd T exercises the half-used last pair)."""
    B, G, K = 2, 2, 2
    NP = G * K
    spec = dict(T=T, dt=0.05, goals=np.zeros((G, 2 * n)), sigma_start_sample=0.05, sigma_gp_sample=0.5, sigma_goal_sample=0.05)
    tab = _tables(spec, cuda)
    sh = _ops().make_shape(B, G, K, S, T, n, dtype, problem_gid0=5)
    mu = torch.zeros(B, NP, T, 2 * n, dtype=dtype, device=cuda)
    x, eps = _ops().sample(sh, tab, mu, seed=0x1234567887654321, draw=3, want_eps=True)
    eps = from_sminor(eps.cpu().numpy())
    want = OPH.normals(0x1234567887654321, 3, 5 * NP + np.arange(B * NP), S, T, n).reshape(B, NP, S, T, 2 * n)
    if dtype == torch.float64:
        assert np.abs(eps - want).max() < 1e-12
    else:
        # fp32 uses the MUFU forms (lg2/sqrt/sin/cos.approx) and rounds (w + 0.5) 2^-32 to 24 bits:
        # |d eps| <~ 5e-6 except in the vanishing-radius corner u1 -> 1
        err = np.abs(eps - want)
        assert np.quantile(err, 0.999) < 2e-5 and err.max() < 5e-3
    _, _, fac = OP.sampling_prior(dict(spec, n_dof=n))
    y = SMP.banded_transform(fac['G'], fac['H'], eps.astype(np.float64))
    assert rel(from_sminor(x.cpu().numpy()), y) < (1e-12 if dtype == torch.float64 else 2e-6)


@pytest.mark.parametrize("dtype,T,n,S,NPg", [(torch.float64, 1024, 7, 512, 4), (torch.float64, 300, 2, 100, 3),
                                              (torch.float32, 512, 14, 64, 2), (torch.float32, 64, 3, 37, 1),
                                              (torch.float64, 200, 5, 520, 40)])
def test_sample_time_chunked_tiles_equal_thread_per_pair(dtype, T, n, S, NPg, cuda):
    """Few samples / long horizons (C5) take the tiled sampler (parallel draw per time chunk, then the recurrence with the state
    carried across chunks); with eps_out requested the thread-per-(sample, DoF pair) kernel runs.  Same stream, same
    expressions: bit-identical samples (ragged S, odd n, chunk counts 1 ... 26, T not a multiple of the chunk)."""
    spec = dict(T=T, dt=0.02, goals=np.zeros((NPg, 2 * n)), sigma_start_sample=0.05, sigma_gp_sample=0.5, sigma_goal_sample=0.05)
    tab = _tables(spec, cuda)
    sh = _ops().make_shape(1, NPg, 1, S, T, n, dtype, problem_gid0=3)
    mu = torch.randn(1, NPg, T, 2 * n, dtype=dtype, device=cuda)
    x_pair, _ = _ops().sample(sh, tab, mu, seed=99, draw=2, want_eps=True)
    x_tile = _ops().sample(sh, tab, mu, seed=99, draw=2)
    assert torch.equal(x_pair, x_tile)


def test_sample_moments_vs_dense_covariance(cuda):
    """Sample covariance of many in-kernel draws against the dense reference covariance P^-1."""
    T, n, S = 6, 1, 200000
    spec = dict(T=T, dt=0.1, goals=np.zeros((1, 2)), sigma_start_sample=0.3, sigma_gp_sample=1.0, sigma_goal_sample=0.3, n_dof=n)
    tab = _tables(spec, cuda)
    sh = _ops().make_shape(1, 1, 1, S, T, n, torch.float64)
    mu = torch.zeros(1, 1, T, 2, dtype=torch.float64, device=cuda)
    x = from_sminor(_ops().sample(sh, tab, mu, seed=7, draw=0).cpu().numpy())[0, 0].reshape(S, -1)
    D, O, _ = OP.sampling_prior(spec)
    Sigma = np.linalg.inv(P.dense_from_blocks(D, O, n))
    C = np.cov(x.T)
    assert np.abs(x.mean(0)).max() < 4 * np.sqrt(np.diag(Sigma).max() / S)
    assert rel(C, Sigma) < 0.02


def test_sample_linearity_full_size(cuda):
    """Size-independent property at the C4 per-particle shape: y(2 eps) = 2 y(eps), y(0) = 0."""
    T, n, S = 64, 7, 512
    spec = dict(T=T, dt=0.05, goals=np.zeros((4, 14)), sigma_start_sample=0.001, sigma_gp_sample=0.1, sigma_goal_sample=0.07)
    tab = _tables(spec, cuda)
    sh = _ops().make_shape(2, 4, 1, S, T, n, torch.float32)
    mu = torch.randn(2, 4, T, 14, device=cuda)
    x1, eps = _ops().sample(sh, tab, mu, seed=1, draw=0, want_eps=True)
    x2 = _ops().sample(sh, tab, mu, eps_in=(2 * eps).contiguous())
    y1 = x1 - mu.unsqueeze(-1)
    y2 = x2 - mu.unsqueeze(-1)
    assert float((y2 - 2 * y1).abs().max() / y1.abs().max()) < 1e-5
    x0 = _ops().sample(sh, tab, mu, eps_in=torch.zeros_like(eps))
    assert torch.equal(x0, mu.unsqueeze(-1).expand_as(x0))


# ---------------------------------------------------------------------------------------------- K3 cost
@pytest.mark.parametrize("name", GOLDEN)
def test_cost_terms_match_reference(name, cuda):
    g = load(name)
    spec = OP.spec_from_golden(g)
    f32 = spec['dtype'] == 'float32'
    dt = torch.float32 if f32 else torch.float64
    pre0 = 'sameL_' if f32 else ''
    tol = TOL_F32 if f32 else FACTOR_TOL_F64.get(name, TOL_F64)
    T = spec['T']
    tab = _tables(spec, cuda)
    _, low = _lowered(spec, cuda, dt)
    sh = _ops().make_shape(1, spec['G'], spec['K'], spec['S'], T, spec['n_dof'], dt)
    sp = torch.tensor(spec['spheres'], device=cuda, dtype=dt).unsqueeze(0) if 'spheres' in spec else None
    D, O, _ = OP.sampling_prior(spec)
    for it in range(n_iters(g, pre0)):
        pre = f'{pre0}it{it}_'
        xs = torch.tensor(to_sminor(g[pre + 'samples']), device=cuda)
        mu = torch.tensor(g[pre + 'means_pre'][None], device=cuda)
        costs, terms = _ops().cost(sh, low.desc(spec['temperature'], sp), tab, xs, mu, want_terms=True)
        terms = terms.cpu().numpy()[:, 0]
        costs = costs.cpu().numpy()[0]
        if pre + 'term_start' in g.files:
            assert rel(terms[0], g[pre + 'term_start']) < tol
        else:
            assert not terms[0].any()                      # CostGPTrajectory: no start factor
        assert rel(terms[0] + terms[1], g[pre + 'term_gp']) < tol
        if 'goals' in g.files and spec['sigma_goal_prior']:
            assert rel(terms[2], g[pre + 'term_goal']) < tol
        if spec['sigma_coll']:
            if 'map' in spec:
                # integer index work: the occupancy sums must be bit-exact
                assert np.array_equal(terms[3], g[pre + 'term_coll'])
            elif 'spheres' in spec:
                assert rel(terms[3], g[pre + 'term_coll']) < (TOL_F32 if f32 else 10 * tol)
        if spec.get('self_margin') is not None:
            assert rel(terms[5], g[pre + 'term_self']) < (TOL_F32 if f32 else 10 * tol)
        if spec.get('ee_target') is not None:
            # fp32: the reference's own fp32 FK + acos carry ~1e-5 of noise on this term (the oracle test allows 1e-4)
            assert rel(terms[6], g[pre + 'term_ee']) < (1e-4 if f32 else 10 * tol)
            ee_o = OP.C.cost_ee_goal(g[pre + 'samples'].astype(np.float64), spec['ee_target'], spec['sigma_ee_goal'], lambda q: OFK.fk_all_links(q),
                                     spec['ee_w_pos'], spec['ee_w_rot'], spec['ee_square'])
            assert rel(terms[6], ee_o) < (TOL_F32 if f32 else 1e-10)
        # IS term: against the fp64 oracle everywhere; against the reference where the reference itself is
        # accurate (fp64).  The fp32 reference's IS term carries up to 4e-3 of cancellation noise.
        _, tot_o = OP.eval_costs(spec, g[pre + 'samples'].astype(np.float64), g[pre + 'means_pre'].astype(np.float64), D, O)
        is_o = OP.C.cost_importance(g[pre + 'samples'].astype(np.float64), g[pre + 'means_pre'].astype(np.float64), D, O, spec['temperature'])
        assert rel(terms[4], is_o) < (TOL_F32 if f32 else 1e-10)
        # fp32 totals vs the fp64 oracle on the same inputs: the north-star's 1e-5
        assert rel(costs, tot_o) < (TOL_F32 if f32 else 1e-10)
        if not f32:
            assert rel(terms[4], g[pre + 'term_is']) < 1e-9
            assert rel(costs, g[pre + 'costs']) < 1e-10
        else:
            assert rel(costs, g[pre + 'costs']) < 1e-2      # bounded by the fp32 reference's own IS-term noise


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("name", GOLDEN_C3)
def test_c3_shape_matches_reference(name, dtype, cuda):
    """The BASELINE shape (4 goals, T = 64, n = 7, S = 256) against a run of the REAL reference at that shape (compact golden:
    the eps are re-drawn from the recorded torch generator state).  fp64: K2 / K3 / the fused iteration against the
    reference's samples, per-term costs, costs, weights, grad and means.  fp32: the reference itself cannot run this shape in
    fp32 (its fp32 Cholesky of the dense precision fails, SURVEY §6), so the fp32 kernels are fed the fp32-rounded inputs and
    held to the north-star's 1e-5 against (i) the fp64 oracle on THE SAME inputs and (ii) the fp64 reference run."""
    g = load(name)
    spec = OP.spec_from_golden(g)
    f32 = dtype == torch.float32
    T, n, G, K, S = spec['T'], spec['n_dof'], spec['G'], spec['K'], spec['S']
    d = 2 * n
    tab = _tables(spec, cuda)
    _, low = _lowered(spec, cuda, dtype)
    sh = _ops().make_shape(1, G, K, S, T, n, dtype)
    sp = torch.tensor(spec['spheres'], device=cuda, dtype=dtype).unsqueeze(0)
    desc = low.desc(spec['temperature'], sp)
    D, O, _ = OP.sampling_prior(spec)
    ftol = 1e-8            # cond(P) ~ 1e9 at T = 64 limits the reference's own dense fp64 factor (tests/test_oracle_golden.py)
    it = 0
    while f'it{it}_rng_state' in g.files:
        pre = f'it{it}_'
        eps_t = eps_ref_to_traj(eps_from_rng_state(g, pre), T, d)                     # [NP, S, T, d] fp64
        eps = torch.tensor(to_sminor(eps_t), device=cuda, dtype=dtype)
        mu = torch.tensor(g[pre + 'means_pre'][None], device=cuda, dtype=dtype)
        xs = _ops().sample(sh, tab, mu, eps_in=eps)
        x = from_sminor(xs.cpu().numpy())[0]
        assert rel(x[:, :2], g[pre + 'samples_head']) < (1e-6 if f32 else ftol)      # fp32: 64 recurrence steps of rounding
        costs, terms = _ops().cost(sh, desc, tab, xs, mu, want_terms=True)
        terms = terms.cpu().numpy()[:, 0]
        costs = costs.cpu().numpy()[0]
        mu_f = mu.clone()
        out = _ops().iterate(sh, desc, tab, spec['step_size'], 1, mu_f, eps_in=eps.unsqueeze(0))
        if not f32:
            assert rel(terms[0] + terms[1], g[pre + 'term_gp']) < 10 * ftol
            assert rel(terms[2], g[pre + 'term_goal']) < 10 * ftol
            assert rel(terms[3], g[pre + 'term_coll']) < 10 * ftol
            assert rel(costs, g[pre + 'costs']) < 10 * ftol
            assert rel(out['costs'].cpu().numpy()[0], g[pre + 'costs']) < 10 * ftol
            assert np.abs(out['weights'].cpu().numpy()[0] - g[pre + 'weights']).max() < 1e-6
            assert rel(out['grad'].cpu().numpy()[0], g[pre + 'grad']) < 1e-5
            assert rel(mu_f.cpu().numpy()[0], g[pre + 'means_post']) < ftol
        else:
            # (i) the fp64 oracle on the SAME fp32-rounded inputs
            r = OP.iterate(spec, mu.cpu().numpy()[0].astype(np.float64), from_sminor(eps.cpu().numpy())[0].astype(np.float64))
            cscale = np.abs(r['costs']).max()
            errs = dict(k3_gp=rel(terms[0] + terms[1], r['terms']['start'] + r['terms']['gp']), k3_goal=rel(terms[2], r['terms']['goal']),
                        k3_coll=rel(terms[3], r['terms']['coll']),
                        # the IS term enters the cost as one summand: its error is measured on the scale of the cost it is added to
                        # (on its own scale the soft case shows 2e-4: sum_t y_t . b_t cancels over the 64 steps in fp32)
                        k3_is_in_cost=float(np.abs(terms[4] - r['terms']['is']).max() / cscale),
                        k3_total=rel(costs, r['costs']), fused_total=rel(out['costs'].cpu().numpy()[0], r['costs']))
            # (ii) against the fp64 reference run on the UNROUNDED inputs: the rounding of the inputs to fp32 is part of this number
            # (the fp64 oracle fed the rounded inputs differs from the reference by `input_rounding`)
            vs_ref = rel(out['costs'].cpu().numpy()[0], g[pre + 'costs'])
            floor = rel(r['costs'], g[pre + 'costs'])
            print(name, it, {k: '%.2e' % v for k, v in errs.items()}, 'fused_vs_reference %.2e input_rounding %.2e' % (vs_ref, floor))
            for k, v in errs.items():
                assert v < TOL_F32, (k, v)
            assert vs_ref < TOL_F32 + floor
            # weights / update: the softmax amplifies cost rounding by |c| / tau, so they are checked on the kernel's OWN costs
            w_o = U_softmax(out['costs'].cpu().numpy()[0].astype(np.float64), spec['temperature'])
            assert np.abs(out['weights'].cpu().numpy()[0] - w_o).max() < 1e-5
        it += 1
    assert it >= 1


@pytest.mark.parametrize("name", GOLDEN_C3)
def test_fused_link_field_term_dominating(name, cuda):
    """The fused role-split kernel evaluates the joint sin/cos of the link warps with MUFU (sin.approx / cos.approx, |err| <= 2^-20.9).
    To see that error where it matters, the cost sigmas are set so that the obstacle term IS the cost (GP / start / goal weights
    ~1e-8 of it): fused fp32 costs against the fp64 oracle on the same inputs, at the north-star's 1e-5, C3 shape."""
    g = load(name)
    spec = dict(OP.spec_from_golden(g), cost_sigma_start=1e3, cost_sigma_gp=1e3, sigma_goal_prior=1e4, sigma_coll=1e-3)
    dtype = torch.float32
    T, n, G, K, S = spec['T'], spec['n_dof'], spec['G'], spec['K'], spec['S']
    d = 2 * n
    tab = _tables(spec, cuda)
    _, low = _lowered(spec, cuda, dtype)
    sh = _ops().make_shape(1, G, K, S, T, n, dtype)
    sp = torch.tensor(spec['spheres'], device=cuda, dtype=dtype).unsqueeze(0)
    desc = low.desc(spec['temperature'], sp)
    pre = 'it0_'
    eps = torch.tensor(to_sminor(eps_ref_to_traj(eps_from_rng_state(g, pre), T, d)), device=cuda, dtype=dtype)
    mu = torch.tensor(g[pre + 'means_pre'][None], device=cuda, dtype=dtype)
    out = _ops().iterate(sh, desc, tab, spec['step_size'], 1, mu.clone(), eps_in=eps.unsqueeze(0))
    r = OP.iterate(spec, mu.cpu().numpy()[0].astype(np.float64), from_sminor(eps.cpu().numpy())[0].astype(np.float64))
    coll_share = float(np.abs(r['terms']['coll']).max() / np.abs(r['costs'] - r['terms']['is']).max())
    assert coll_share > 0.99                                     # the obstacle term really is the cost here
    cost_wo_is = out['costs'].cpu().numpy()[0].astype(np.float64) - r['terms']['is']
    err = rel(cost_wo_is, r['costs'] - r['terms']['is'])
    print(name, 'link-field-dominated cost: fused fp32 vs fp64 oracle %.2e' % err)
    assert err < TOL_F32


def U_softmax(costs, tau):
    z = -costs / tau
    z = z - z.max(-1, keepdims=True)
    e = np.exp(z)
    return e / e.sum(-1, keepdims=True)


def test_cost_eval_dropin(cuda):
    """CostComposite.eval(trajs) on CUDA tensors == sum of the reference's cost terms (no IS term)."""
    g = load('planar_f64')
    spec = OP.spec_from_golden(g)
    comp, _ = _lowered(spec, cuda, torch.float64)
    x = torch.tensor(g['it0_samples'], device=cuda)
    got = comp.eval(x).cpu().numpy().reshape(g['it0_costs'].shape)
    want = g['it0_term_gp'] + g['it0_term_goal'] + g['it0_term_coll']
    assert rel(got, want) < 1e-12
    # single cost objects
    assert rel(comp.cost_list[0].eval(x.reshape(-1, spec['T'], 4)).cpu().numpy().reshape(want.shape), g['it0_term_gp']) < 1e-12


def test_map_lookup_edges(cuda):
    """Out-of-range points clamp to the border, value = map[iy][ix] (obst_map.py:173-181); fp32 and fp64."""
    from stoch_gpmp_b200.envs.occupancy import ObstacleMap
    from oracle import costs as C
    rs = np.random.RandomState(0)
    for dtype, npdt in ((torch.float32, np.float32), (torch.float64, np.float64)):
        om = ObstacleMap([4, 4], 0.1, tensor_args=dict(device=cuda, dtype=dtype))
        om.map = rs.randint(0, 3, om.map.shape).astype(np.float64)
        xy = np.concatenate([rs.uniform(-3, 3, (4000, 2)), np.array([[-2.0, -2.0], [2.0, 2.0], [1.95, -1.95], [0.0, 0.0], [0.1, 0.2], [-0.1, 0.3]])]).astype(npdt)
        got = om.compute_cost(torch.tensor(xy, device=cuda)).cpu().numpy()
        want = C.map_lookup(xy, om.map.astype(npdt), 0.1, om.origin_xi, om.origin_yi)
        assert np.array_equal(got, want)


def test_fk_known_answers_cuda(cuda):
    from stoch_gpmp_b200.robots import PandaFK
    fk = PandaFK()
    q = torch.tensor([[0.] * 7, [0.012, -0.57, 0., -2.81, 0., 3.037, 0.741]], dtype=torch.float64, device=cuda)
    pos = _ops().fk_link_positions(fk, q).cpu().numpy()
    assert pos.shape == (2, 11, 3)
    assert np.allclose(pos[0, 8], [0.088, 0.0, 0.926], atol=1e-9)
    assert np.allclose(pos[0, 10], [0.088, 0.0, 0.826], atol=1e-9)
    assert np.allclose(pos[1, 10], [0.460816, 0.005530, 0.388328], atol=2e-6)
    rs = np.random.RandomState(1)
    qr = rs.uniform(-2.8, 2.8, (257, 7))
    want = OFK.fk_all_links(qr)[:, :, :3, 3]
    assert rel(_ops().fk_link_positions(fk, torch.tensor(qr, device=cuda)).cpu().numpy(), want) < 1e-13
    assert rel(_ops().fk_link_positions(fk, torch.tensor(qr, device=cuda, dtype=torch.float32)).cpu().numpy(), want) < 2e-6


# -------------------------------------------------------------------------------------------- K4 update
@pytest.mark.parametrize("name", GOLDEN)
def test_update_matches_reference(name, cuda):
    """Feed the REFERENCE's costs and samples: weights, grad and new means must match."""
    g = load(name)
    spec = OP.spec_from_golden(g)
    f32 = spec['dtype'] == 'float32'
    dt = torch.float32 if f32 else torch.float64
    pre0 = 'sameL_' if f32 else ''
    sh = _ops().make_shape(1, spec['G'], spec['K'], spec['S'], spec['T'], spec['n_dof'], dt)
    for it in range(n_iters(g, pre0)):
        pre = f'{pre0}it{it}_'
        xs = torch.tensor(to_sminor(g[pre + 'samples']), device=cuda)
        mu = torch.tensor(g[pre + 'means_pre'][None], device=cuda).clone()
        c = torch.tensor(g[pre + 'costs'][None], device=cuda)
        grad, w = _ops().update(sh, spec['temperature'], spec['step_size'], c, xs, mu)
        assert np.abs(w.cpu().numpy()[0] - g[pre + 'weights']).max() < (1e-5 if f32 else 1e-12)
        assert rel(grad.cpu().numpy()[0], g[pre + 'grad']) < (TOL_F32 if f32 else 1e-10)
        assert rel(mu.cpu().numpy()[0], g[pre + 'means_post']) < (1e-6 if f32 else 1e-12)


# ------------------------------------------------------------------------------------------ fused loop
@pytest.mark.parametrize("name", GOLDEN)
def test_fused_iteration_matches_reference(name, cuda):
    """sgpmp_iterate with the reference's eps: samples, costs, weights, grad, means — chained iterations."""
    g = load(name)
    spec = OP.spec_from_golden(g)
    f32 = spec['dtype'] == 'float32'
    dt = torch.float32 if f32 else torch.float64
    pre0 = 'sameL_' if f32 else ''
    ftol = TOL_F32 if f32 else FACTOR_TOL_F64.get(name, TOL_F64)
    T, d = spec['T'], 2 * spec['n_dof']
    tab = _tables(spec, cuda)
    _, low = _lowered(spec, cuda, dt)
    sh = _ops().make_shape(1, spec['G'], spec['K'], spec['S'], T, spec['n_dof'], dt)
    sp = torch.tensor(spec['spheres'], device=cuda, dtype=dt).unsqueeze(0) if 'spheres' in spec else None
    D, O, _ = OP.sampling_prior(spec)
    for it in range(n_iters(g, pre0)):
        pre = f'{pre0}it{it}_'
        eps = torch.tensor(to_sminor(eps_ref_to_traj(g[pre + 'eps'], T, d)), device=cuda).unsqueeze(0).contiguous()
        mu = torch.tensor(g[pre + 'means_pre'][None], device=cuda).clone()
        out = _ops().iterate(sh, low.desc(spec['temperature'], sp), tab, spec['step_size'], 1, mu, eps_in=eps, want_samples=True)
        assert np.array_equal(out['means_pre'].cpu().numpy()[0], g[pre + 'means_pre'])
        assert rel(from_sminor(out['samples'].cpu().numpy())[0], g[pre + 'samples']) < ftol
        costs = out['costs'].cpu().numpy()[0]
        if not f32:
            assert rel(costs, g[pre + 'costs']) < max(ftol, 1e-10)
            assert np.abs(out['weights'].cpu().numpy()[0] - g[pre + 'weights']).max() < 1e-7
            assert rel(out['grad'].cpu().numpy()[0], g[pre + 'grad']) < max(10 * ftol, 1e-9)
            assert rel(mu.cpu().numpy()[0], g[pre + 'means_post']) < ftol
        else:
            # fp32: total costs vs the accurate (fp64) oracle; weights/update from the kernel's own costs
            r = OP.iterate(spec, g[pre + 'means_pre'], eps_ref_to_traj(g[pre + 'eps'], T, d))
            assert rel(costs, r['costs']) < 3e-5      # fp32 rounding floor of the GP term, see test_cost_terms_match_reference
            from oracle import update as U
            mp, grad, w = U.update(g[pre + 'means_pre'].astype(np.float64), r['samples'], costs.astype(np.float64),
                                   spec['temperature'], spec['step_size'])
            assert np.abs(out['weights'].cpu().numpy()[0] - w).max() < 1e-5
            assert rel(out['grad'].cpu().numpy()[0], grad) < 2e-5
            assert rel(mu.cpu().numpy()[0], mp) < 1e-6


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("case", ["planar", "panda"])
def test_fused_equals_separate_kernels_inkernel_rng(case, dtype, cuda):
    """Fused loop (in-kernel Philox, 3 iterations in one launch) == K2 -> K3 -> K4 chained with the same
    draw indices.  Soft sigmas so that many samples carry weight (exercises the weighted eps-sum pass)."""
    g = load('planar_soft_f64' if case == 'planar' else 'panda_soft_f64')
    spec = OP.spec_from_golden(g)
    B, S = 3, 96 if case == 'planar' else 40
    spec = dict(spec, S=S)
    T, n, G, K = spec['T'], spec['n_dof'], spec['G'], spec['K']
    tab = _tables(spec, cuda)
    _, low = _lowered(spec, cuda, dtype, B=B)
    sp = torch.tensor(spec['spheres'], device=cuda, dtype=dtype).unsqueeze(0) if 'spheres' in spec else None
    desc = low.desc(spec['temperature'], sp)
    sh = _ops().make_shape(B, G, K, S, T, n, dtype, problem_gid0=11)
    mu0 = torch.tensor(g['it0_means_pre'], device=cuda, dtype=dtype).unsqueeze(0).repeat(B, 1, 1, 1).contiguous()
    mu0 += 0.01 * torch.arange(B, device=cuda, dtype=dtype).view(B, 1, 1, 1)
    # The loop is chaotic in fp32 (a mean perturbation d changes the logits by ~|dc/dmu| d / tau ~ 200 d here), so
    # the two paths are compared iteration by iteration from the SAME means; fp64 also checks the 3-iteration chain.
    # fp32: the fused kernel sums per-DoF-pair partial costs (packed FP32), K3 sums serially: 4e-5 apart on costs of
    # ~6e4 that cancel from larger terms; both are within 1e-5 of the fp64 oracle on the golden cases.
    tol = 1e-4 if dtype == torch.float32 else 1e-9
    wtol = 2e-3 if dtype == torch.float32 else 1e-8
    mu_s = mu0.clone()
    for it in range(3):
        pre_means = mu_s.clone()
        mu_f = mu_s.clone()
        out = _ops().iterate(sh, desc, tab, spec['step_size'], 1, mu_f, seed=99, draw0=4 + it, want_samples=True)
        xs = _ops().sample(sh, tab, mu_s, seed=99, draw=4 + it)
        c = _ops().cost(sh, desc, tab, xs, mu_s)
        grad, w = _ops().update(sh, spec['temperature'], spec['step_size'], c, xs, mu_s)
        assert torch.equal(out['means_pre'], pre_means)
        assert float((out['samples'] - xs).abs().max() / xs.abs().max()) < (2e-6 if dtype == torch.float32 else tol)
        assert float((out['costs'] - c).abs().max() / c.abs().max()) < tol
        assert float((out['weights'] - w).abs().max()) < wtol
        assert float((out['grad'] - grad).abs().max() / grad.abs().max()) < 10 * wtol
        assert float((mu_f - mu_s).abs().max() / mu_s.abs().max()) < 10 * wtol
    if dtype == torch.float64:
        mu_c = mu0.clone()
        outc = _ops().iterate(sh, desc, tab, spec['step_size'], 3, mu_c, seed=99, draw0=4, want_samples=True)
        assert float((mu_c - mu_s).abs().max() / mu_s.abs().max()) < 1e-7
        assert float((outc['costs'] - c).abs().max() / c.abs().max()) < 1e-7
    ess = 1.0 / (w.double() ** 2).sum(-1)
    assert float(ess.max()) > 1.5          # the weighted pass really was exercised


@pytest.mark.parametrize("n", [5, 14])
def test_fused_iteration_other_dof_counts(n, cuda):
    """n_dof 5 and 14 (the DoF counts of BASELINE's C5 sweep that round 1 could only sample): the fused loop against the
    numpy oracle on the kernel's own eps (GP + goal factors; the reference is generic in n_dof, planner.py:51-52), fp64."""
    from stoch_gpmp_b200.costs.cost_functions import CostComposite, CostGP, CostGoalPrior
    dtype = torch.float64
    T, G, K, S, B = 12, 2, 1, 40, 2
    d = 2 * n
    ta = dict(device=cuda, dtype=dtype)
    rs = np.random.RandomState(n)
    start = rs.uniform(-0.3, 0.3, (B, d))
    goals = rs.uniform(-0.5, 0.5, (B, G, d))
    spec = dict(n_dof=n, T=T, dt=0.1, G=G, K=K, S=S, temperature=20.0, step_size=0.5, goals=goals[0], start=start[0],
                sigma_start_sample=0.3, sigma_gp_sample=1.0, sigma_goal_sample=0.3, cost_sigma_start=0.5, cost_sigma_gp=2.0,
                sigma_goal_prior=1.0, sigma_coll=None)
    tab = _tables(spec, cuda)
    comp = CostComposite(n, T, [CostGP(n, T, torch.tensor(start, **ta), 0.1, dict(sigma_start=0.5, sigma_gp=2.0), ta),
                                CostGoalPrior(n, T, multi_goal_states=torch.tensor(goals, **ta), num_particles_per_goal=K, num_samples=S,
                                              sigma_goal_prior=1.0, tensor_args=ta)], tensor_args=ta)
    desc = comp.lower(B, G, cuda, dtype).desc(20.0, None)
    sh = _ops().make_shape(B, G, K, S, T, n, dtype)
    mu = torch.tensor(rs.uniform(-0.5, 0.5, (B, G * K, T, d)), **ta)
    mu_f = mu.clone()
    out = _ops().iterate(sh, desc, tab, 0.5, 1, mu_f, seed=5, draw0=2)
    _, eps = _ops().sample(sh, tab, mu, seed=5, draw=2, want_eps=True)
    eps = from_sminor(eps.cpu().numpy())
    for b in range(B):
        r = OP.iterate(dict(spec, start=start[b], goals=goals[b]), mu[b].cpu().numpy(), eps[b])
        assert rel(out['costs'][b].cpu().numpy(), r['costs']) < 1e-10
        assert rel(mu_f[b].cpu().numpy(), r['means_post']) < 1e-10


def test_fused_problem_sharding_invariance(cuda):
    """B problems in one launch == the same problems launched as two shards with problem_gid0 offsets."""
    g = load('panda_soft_f32')
    spec = dict(OP.spec_from_golden(g), S=64)
    T, n, G, K, S = spec['T'], spec['n_dof'], spec['G'], spec['K'], spec['S']
    B = 4
    dtype = torch.float32
    tab = _tables(spec, cuda)
    rs = np.random.RandomState(3)
    starts = torch.tensor(spec['start'][None] + 0.05 * rs.randn(B, 2 * n), device=cuda, dtype=dtype)
    goals = torch.tensor(spec['goals'][None] + 0.05 * rs.randn(B, G, 2 * n), device=cuda, dtype=dtype)
    spheres = torch.tensor(spec['spheres'][None] + 0.02 * rs.randn(B, len(spec['spheres']), 4), device=cuda, dtype=dtype)
    mu0 = torch.tensor(g['it0_means_pre'], device=cuda, dtype=dtype).unsqueeze(0).repeat(B, 1, 1, 1).contiguous()

    def run(lo, hi):
        from stoch_gpmp_b200.costs.cost_functions import CostCollision, CostComposite, CostGP, CostGoalPrior
        from stoch_gpmp_b200.costs.fields import LinkDistanceField
        from stoch_gpmp_b200.robots import PandaFK
        ta = dict(device=cuda, dtype=dtype)
        comp = CostComposite(n, T, [
            CostGP(n, T, starts[lo:hi], spec['dt'], dict(sigma_start=spec['cost_sigma_start'], sigma_gp=spec['cost_sigma_gp']), ta),
            CostGoalPrior(n, T, multi_goal_states=goals[lo:hi], num_particles_per_goal=K, num_samples=S,
                          sigma_goal_prior=spec['sigma_goal_prior'], tensor_args=ta),
            CostCollision(n, T, field=LinkDistanceField(tensor_args=ta), sigma_coll=spec['sigma_coll'])], FK=PandaFK(), tensor_args=ta)
        low = comp.lower(hi - lo, G, cuda, dtype)
        sh = _ops().make_shape(hi - lo, G, K, S, T, n, dtype, problem_gid0=lo)
        mu = mu0[lo:hi].clone()
        out = _ops().iterate(sh, low.desc(spec['temperature'], spheres[lo:hi].contiguous()), tab, spec['step_size'], 2, mu, seed=5, draw0=0)
        return mu, out['costs']
    mu_all, c_all = run(0, B)
    mu_a, c_a = run(0, 1)
    mu_b, c_b = run(1, B)
    assert torch.equal(mu_all, torch.cat([mu_a, mu_b]))
    assert torch.equal(c_all, torch.cat([c_a, c_b]))


def test_fused_full_size_properties(cuda):
    """C4 per-problem shape (G=4, K=1, S=512, T=64, n=7, fp32) on a few problems: size-independent
    properties — weights sum to one, grad == sum_s w_s (x_s - mu) on the emitted samples (K4 on the fused
    kernel's own outputs), determinism, and emitted costs == K3 on the emitted samples.  12 particles with S=512 run the
    single-role kernel in clusters of 8 CTAs (the role-split kernel at this per-problem shape is test_gpu_fused_shapes case d)."""
    from test_gpu_fused_shapes import expect_kernel
    T, n, G, K, S, B = 64, 7, 4, 1, 512, 3
    dtype = torch.float32
    rs = np.random.RandomState(0)
    from stoch_gpmp_b200.scenarios import PANDA_START, panda_goals, panda_spheres
    spec = dict(n_dof=n, T=T, dt=0.05, G=G, K=K, S=S, temperature=1.0, step_size=0.1, start=np.array(PANDA_START),
                goals=np.array(panda_goals(G, 3)), cost_sigma_start=1e-4, cost_sigma_gp=7e-4, sigma_goal_prior=20., sigma_coll=0.01,
                spheres=np.array(panda_spheres(5, 3)), sigma_start_sample=1e-3, sigma_gp_sample=0.1, sigma_goal_sample=0.07)
    tab = _tables(spec, cuda)
    _, low = _lowered(spec, cuda, dtype, B=B)
    sp = torch.tensor(spec['spheres'], device=cuda, dtype=dtype).unsqueeze(0)
    sh = _ops().make_shape(B, G, K, S, T, n, dtype)
    from stoch_gpmp_b200.planner import StochGPMPBatch  # noqa: F401  (import check)
    mu0 = torch.tensor(P.const_vel_trajectories(spec['start'], spec['goals'], 0.05, T, n, K).reshape(1, G * K, T, 2 * n),
                       device=cuda, dtype=dtype).repeat(B, 1, 1, 1).contiguous()
    res = []
    for rep in range(2):
        mu = mu0.clone()
        with expect_kernel(r"iterate_kernel<float, ?2, ?7, ?64, ?1, ?8>"):
            out = _ops().iterate(sh, low.desc(1.0, sp), tab, 0.1, 1, mu, seed=1, draw0=0, want_samples=True)
        res.append((mu, out))
    (mu1, o1), (mu2, o2) = res
    for k in ('samples', 'costs', 'weights', 'grad'):
        assert torch.equal(o1[k], o2[k])
    assert torch.equal(mu1, mu2)
    assert float((o1['weights'].sum(-1) - 1).abs().max()) < 1e-5
    c3 = _ops().cost(sh, low.desc(1.0, sp), tab, o1['samples'], mu0)
    assert float((c3 - o1['costs']).abs().max() / c3.abs().max()) < 1e-5
    mu_k4 = mu0.clone()
    grad, w = _ops().update(sh, 1.0, 0.1, o1['costs'], o1['samples'], mu_k4)
    assert float((w - o1['weights']).abs().max()) < 1e-6
    assert float((grad - o1['grad']).abs().max() / grad.abs().max()) < 1e-4
    assert float((mu_k4 - mu1).abs().max() / mu1.abs().max()) < 1e-6


# ---------------------------------------------------------------------------------------- split mode
def test_split_particle_stats_equal_single_update(cuda):
    """One problem's samples split in two halves: local stats -> log-sum-exp merge -> apply == K4 on all."""
    g = load('planar_soft_f64')
    spec = OP.spec_from_golden(g)
    T, n, G, K, S = spec['T'], spec['n_dof'], spec['G'], spec['K'], spec['S']
    dt = torch.float64
    tab = _tables(spec, cuda)
    eps = torch.tensor(to_sminor(eps_ref_to_traj(g['it0_eps'], T, 2 * n)), device=cuda)
    xs = torch.tensor(to_sminor(g['it0_samples']), device=cuda)
    c = torch.tensor(g['it0_costs'][None], device=cuda)
    mu = torch.tensor(g['it0_means_pre'][None], device=cuda)
    sh = _ops().make_shape(1, G, K, S, T, n, dt)
    mu_ref = mu.clone()
    grad_ref, _ = _ops().update(sh, spec['temperature'], spec['step_size'], c, xs, mu_ref)
    h = S // 2
    shh = _ops().make_shape(1, G, K, h, T, n, dt)
    st = [_ops().local_stats(shh, spec['temperature'], c[..., a:a + h].contiguous(), eps[..., a:a + h].contiguous()) for a in (0, h)]
    merged = _ops().merge_stats(st).contiguous()
    mu_split = mu.clone()
    grad = _ops().apply_stats(sh, tab, spec['step_size'], merged, mu_split)
    assert rel(grad.cpu().numpy(), grad_ref.cpu().numpy()) < 1e-9
    assert rel(mu_split.cpu().numpy(), mu_ref.cpu().numpy()) < 1e-12
    assert rel(mu_split.cpu().numpy()[0], g['it0_means_post']) < 1e-10


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("n,T,S,G,K", [(2, 7, 33, 1, 3), (3, 9, 5, 2, 1), (4, 6, 130, 1, 1), (6, 5, 17, 2, 2), (7, 11, 257, 1, 1)])
def test_fused_ragged_shapes_equal_separate_kernels(n, T, S, G, K, dtype, cuda):
    """Edge shapes through the fused loop — odd T (half-used last Philox pair), odd S, S not a multiple of the
    block size, one sample chunk more than a block, every instantiated DoF count (odd n exercises the ghost DoF
    of the packed kernel), a single goal — against K2 -> K3 -> K4 with the same draw index."""
    from stoch_gpmp_b200.costs.cost_functions import CostComposite, CostGP, CostGoalPrior
    B = 2
    d = 2 * n
    ta = dict(device=cuda, dtype=dtype)
    rs = np.random.RandomState(n * 100 + T)
    spec = dict(T=T, dt=0.1, goals=np.zeros((G, d)), sigma_start_sample=0.3, sigma_gp_sample=1.0, sigma_goal_sample=0.3)
    tab = _tables(spec, cuda)
    start = torch.tensor(rs.uniform(-0.3, 0.3, (B, d)), **ta)
    goals = torch.tensor(rs.uniform(-0.5, 0.5, (B, G, d)), **ta)
    comp = CostComposite(n, T, [CostGP(n, T, start, 0.1, dict(sigma_start=0.5, sigma_gp=2.0), ta),
                                CostGoalPrior(n, T, multi_goal_states=goals, num_particles_per_goal=K, num_samples=S,
                                              sigma_goal_prior=1.0, tensor_args=ta)], tensor_args=ta)
    low = comp.lower(B, G, cuda, dtype)
    desc = low.desc(20.0, None)
    sh = _ops().make_shape(B, G, K, S, T, n, dtype, problem_gid0=3)
    mu0 = torch.tensor(rs.uniform(-0.5, 0.5, (B, G * K, T, d)), **ta)
    mu_f, mu_s = mu0.clone(), mu0.clone()
    out = _ops().iterate(sh, desc, tab, 0.5, 1, mu_f, seed=17, draw0=2, want_samples=True)
    xs = _ops().sample(sh, tab, mu_s, seed=17, draw=2)
    c = _ops().cost(sh, desc, tab, xs, mu_s)
    grad, w = _ops().update(sh, 20.0, 0.5, c, xs, mu_s)
    f32 = dtype == torch.float32
    assert float((out['samples'] - xs).abs().max() / xs.abs().max()) < (2e-6 if f32 else 1e-12)
    assert float((out['costs'] - c).abs().max() / c.abs().max()) < (2e-5 if f32 else 1e-11)
    assert float((out['weights'] - w).abs().max()) < (1e-4 if f32 else 1e-10)
    assert float((out['grad'] - grad).abs().max() / grad.abs().max()) < (1e-3 if f32 else 1e-9)
    assert float((mu_f - mu_s).abs().max() / mu_s.abs().max()) < (1e-4 if f32 else 1e-10)
    assert float((out['weights'].sum(-1) - 1).abs().max()) < 1e-5


@pytest.mark.parametrize("name,R", [("panda_soft_f64", 4), ("panda_soft_f32", 2), ("planar_soft_f64", 8), ("panda_self_f32", 4)])
def test_split_particle_fused_equals_fused_iterate(name, R, cuda):
    """Split-particle mode emulated on ONE GPU: R 'ranks' run sgpmp_iterate_stats over their slices of every particle's samples
    (global sample ids keep the RNG stream), the R (m, Z, A) blocks are merged by log-sum-exp INSIDE sgpmp_merge_apply_stats,
    and the resulting means equal the single-launch fused iteration on all samples (planner.py:263-275 is what is being split).
    The same code with ncclAllGather between the two launches is tests/test_gpu_multi.py / bench.py --gpus N."""
    g = load(name)
    spec = OP.spec_from_golden(g)
    f32 = spec['dtype'] == 'float32'
    dt = torch.float32 if f32 else torch.float64
    T, n, G, K, S = spec['T'], spec['n_dof'], spec['G'], spec['K'], spec['S']
    assert S % R == 0
    tab = _tables(spec, cuda)
    _, low = _lowered(spec, cuda, dt)
    sp = torch.tensor(spec['spheres'], device=cuda, dtype=dt).unsqueeze(0) if 'spheres' in spec else None
    desc = low.desc(spec['temperature'], sp)
    pre = 'sameL_' if f32 else ''
    mu = torch.tensor(g[pre + 'it0_means_pre'][None], device=cuda)
    sh = _ops().make_shape(1, G, K, S, T, n, dt)
    for it in range(2):
        mu_f = mu.clone()
        out = _ops().iterate(sh, desc, tab, spec['step_size'], 1, mu_f, seed=29, draw0=it)
        stats, costs = [], []
        for r in range(R):
            shr = _ops().make_shape(1, G, K, S // R, T, n, dt, sample_gid0=r * (S // R))
            st, c = _ops().iterate_stats(shr, desc, tab, mu, seed=29, draw=it, want_costs=True)
            stats.append(st)
            costs.append(c)
        c_all = torch.cat(costs, dim=-1)
        assert float((c_all - out['costs']).abs().max() / out['costs'].abs().max()) < (1e-6 if f32 else 1e-13)
        mu_s = mu.clone()
        grad = _ops().merge_apply_stats(sh, tab, spec['step_size'], torch.stack(stats, 0).contiguous(), mu_s)
        # the softmax amplifies fp32 cost rounding (|c|/tau up to 1e2..1e3 in the soft goldens): fp32 is held to 1e-4
        assert float((grad - out['grad']).abs().max() / out['grad'].abs().max()) < (1e-3 if f32 else 1e-9)
        assert float((mu_s - mu_f).abs().max() / mu_f.abs().max()) < (1e-4 if f32 else 1e-10)
        # the torch restatement of the merge (parallel.allreduce_stats, used by the gloo CPU test) agrees with the kernel
        mu_t = mu.clone()
        _ops().apply_stats(sh, tab, spec['step_size'], _ops().merge_stats(stats).contiguous(), mu_t)
        assert float((mu_t - mu_s).abs().max() / mu_s.abs().max()) < (1e-6 if f32 else 1e-13)
        mu = mu_f
    # n iterations enqueued by ONE call of the split-mode driver with a single rank == the fused loop
    mu_a = torch.tensor(g[pre + 'it0_means_pre'][None], device=cuda)
    mu_b = mu_a.clone()
    o = _ops().iterate_split_particles(sh, desc, tab, spec['step_size'], 3, mu_a, 29, 0)
    _ops().iterate(sh, desc, tab, spec['step_size'], 3, mu_b, seed=29, draw0=0)
    assert float((mu_a - mu_b).abs().max() / mu_b.abs().max()) < (2e-3 if f32 else 1e-9)
    assert o['means_pre'] is not None and o['costs'].shape == (1, G * K, S)


@pytest.mark.parametrize("n,S", [(2, 512), (7, 256), (7, 300)])
def test_cluster_mode_equals_separate_kernels(n, S, cuda):
    """Few problems (B*NP*8 <= 296 CTAs) with S >= 256 run the fused loop in thread-block-CLUSTER mode: a particle's
    samples are split over 8 CTAs and the softmax / weighted-sum reductions go through distributed shared memory.
    The result must equal K2 -> K3 -> K4 (no clusters) on the same draw; S=300 leaves ragged per-CTA slices."""
    from stoch_gpmp_b200.costs.cost_functions import CostComposite, CostGP, CostGoalPrior
    dtype = torch.float32
    B, G, K, T = 1, 3, 1, 16
    d = 2 * n
    ta = dict(device=cuda, dtype=dtype)
    rs = np.random.RandomState(n + S)
    spec = dict(T=T, dt=0.1, goals=np.zeros((G, d)), sigma_start_sample=0.3, sigma_gp_sample=1.0, sigma_goal_sample=0.3)
    tab = _tables(spec, cuda)
    start = torch.tensor(rs.uniform(-0.3, 0.3, (B, d)), **ta)
    goals = torch.tensor(rs.uniform(-0.5, 0.5, (B, G, d)), **ta)
    comp = CostComposite(n, T, [CostGP(n, T, start, 0.1, dict(sigma_start=0.5, sigma_gp=2.0), ta),
                                CostGoalPrior(n, T, multi_goal_states=goals, num_particles_per_goal=K, num_samples=S,
                                              sigma_goal_prior=1.0, tensor_args=ta)], tensor_args=ta)
    desc = comp.lower(B, G, cuda, dtype).desc(20.0, None)
    sh = _ops().make_shape(B, G, K, S, T, n, dtype)
    mu0 = torch.tensor(rs.uniform(-0.5, 0.5, (B, G * K, T, d)), **ta)
    # fp32 softmax amplifies cost rounding (|c|/tau ~ 1e2..1e3 here), so the update is checked on the kernel's OWN costs:
    # K4 fed the fused kernel's costs and K2's samples of the same draw must reproduce its weights and means.
    mu = mu0.clone()
    for it in range(2):
        xs = _ops().sample(sh, tab, mu, seed=23, draw=it)
        c = _ops().cost(sh, desc, tab, xs, mu)
        mu_f = mu.clone()
        out = _ops().iterate(sh, desc, tab, 0.5, 1, mu_f, seed=23, draw0=it, want_samples=True)
        assert torch.equal(out['means_pre'], mu)
        assert float((out['samples'] - xs).abs().max() / xs.abs().max()) < 2e-6
        assert float((out['costs'] - c).abs().max() / c.abs().max()) < 1e-4
        mu_k = mu.clone()
        grad, w = _ops().update(sh, 20.0, 0.5, out['costs'], xs, mu_k)
        assert float((out['weights'] - w).abs().max()) < 1e-5
        assert float((out['grad'] - grad).abs().max() / grad.abs().max()) < 1e-4
        assert float((mu_f - mu_k).abs().max() / mu_k.abs().max()) < 1e-5
        assert float((out['weights'].sum(-1) - 1).abs().max()) < 1e-5
        mu = mu_f
    # two iterations inside ONE cluster launch == two single-iteration launches
    mu_2 = mu0.clone()
    _ops().iterate(sh, desc, tab, 0.5, 2, mu_2, seed=23, draw0=0)
    assert torch.equal(mu_2, mu)


@pytest.mark.parametrize("T,n,S", [(128, 4, 4096), (256, 14, 2048), (1024, 2, 2048), (1024, 14, 512)])
def test_c5_sampling_sweep_fp64(T, n, S, cuda):
    """BASELINE configs[4]: prior construction + sampling for long horizons / many DoF in fp64 (the reference would
    need a dense M x M factor per particle: M = 28,672 -> 6.6 GB at T=1024, n=14).  Checks: (i) the kernel's
    samples equal the oracle recurrence on the kernel's own eps; (ii) per-DoF sample moments against the dense
    2T x 2T covariance (valid because the precision decouples per DoF) where that inverse is cheap."""
    spec = dict(T=T, dt=0.02, goals=np.zeros((1, 2 * n)), sigma_start_sample=1e-3, sigma_gp_sample=3.0, sigma_goal_sample=1e-3, n_dof=n)
    tab = _tables(spec, cuda)
    D, O = P.precision_blocks(T, 0.02, 1e-3, 3.0, 1e-3)
    fac = P.banded_factor(D, O)
    sh = _ops().make_shape(1, 1, 1, S, T, n, torch.float64)
    mu = torch.zeros(1, 1, T, 2 * n, dtype=torch.float64, device=cuda)
    x, eps = _ops().sample(sh, tab, mu, seed=5, draw=0, want_eps=True)
    x = from_sminor(x.cpu().numpy())[0, 0]              # [S, T, d]
    e = from_sminor(eps.cpu().numpy())[0, 0]
    sub = slice(0, 64)
    y = SMP.banded_transform(fac['G'], fac['H'], e[sub])
    assert rel(x[sub], y) < 1e-12
    if T <= 256:
        Sigma = np.linalg.inv(P.dense_from_blocks(D, O, 1))
        sd = np.sqrt(np.diag(Sigma))
        # pool the n DoFs: S*n independent draws of the same 2T-dimensional Gaussian
        z = np.concatenate([np.concatenate([x[:, :, i:i + 1], x[:, :, n + i:n + i + 1]], axis=2).reshape(S, 2 * T) for i in range(n)])
        C = np.cov(z.T)
        corr_err = np.abs(C - Sigma) / np.outer(sd, sd)
        assert corr_err.max() < 6.0 / np.sqrt(z.shape[0])
        assert np.abs(z.mean(0) / sd).max() < 5.0 / np.sqrt(z.shape[0])
    else:
        # long horizon: marginal variances against the diagonal of Sigma obtained from the factor itself (L L^T)
        var = x.reshape(S, T, 2, n).var(axis=(0, 3))
        Ld = P.dense_scale_tril(fac['G'], fac['H'], 1) if T <= 1024 else None
        diag = (Ld ** 2).sum(1).reshape(T, 2)
        assert np.abs(var / diag - 1).max() < 8.0 / np.sqrt(S * n)


@pytest.mark.parametrize("B,S", [(2, 512), (6, 256), (12, 192), (20, 128)])
def test_cluster_sizes_agree_with_one_problem_at_a_time(B, S, cuda):
    """The cluster size (8 / 4 / 2 / 1) is chosen from the number of particles and samples; a batch of B problems
    must give, per problem, what that problem gives when launched alone (which uses the largest cluster)."""
    from stoch_gpmp_b200.costs.cost_functions import CostComposite, CostGP, CostGoalPrior
    n, T, G, K = 7, 8, 4, 1
    d = 2 * n
    dtype = torch.float32
    ta = dict(device=cuda, dtype=dtype)
    rs = np.random.RandomState(B)
    spec = dict(T=T, dt=0.1, goals=np.zeros((G, d)), sigma_start_sample=0.3, sigma_gp_sample=1.0, sigma_goal_sample=0.3)
    tab = _tables(spec, cuda)
    start = torch.tensor(rs.uniform(-0.3, 0.3, (B, d)), **ta)
    goals = torch.tensor(rs.uniform(-0.5, 0.5, (B, G, d)), **ta)
    mu0 = torch.tensor(rs.uniform(-0.5, 0.5, (B, G * K, T, d)), **ta)

    def run(lo, hi):
        comp = CostComposite(n, T, [CostGP(n, T, start[lo:hi], 0.1, dict(sigma_start=0.5, sigma_gp=2.0), ta),
                                    CostGoalPrior(n, T, multi_goal_states=goals[lo:hi], num_particles_per_goal=K, num_samples=S,
                                                  sigma_goal_prior=1.0, tensor_args=ta)], tensor_args=ta)
        desc = comp.lower(hi - lo, G, cuda, dtype).desc(20.0, None)
        sh = _ops().make_shape(hi - lo, G, K, S, T, n, dtype, problem_gid0=lo)
        mu = mu0[lo:hi].clone()
        out = _ops().iterate(sh, desc, tab, 0.5, 2, mu, seed=3, draw0=0)
        return mu, out['costs']
    mu_all, c_all = run(0, B)
    for b in (0, B - 1):
        mu_b, c_b = run(b, b + 1)
        assert float((c_all[b] - c_b[0]).abs().max() / c_b.abs().max()) < 1e-5
        assert float((mu_all[b] - mu_b[0]).abs().max() / mu_b.abs().max()) < 1e-3       # fp32 softmax sensitivity


# ------------------------------------------------------------------------ weighted covariance (tensor cores)
@pytest.mark.parametrize("n,T,S,NP", [(7, 64, 512, 2), (2, 64, 256, 3), (7, 10, 40, 2), (3, 7, 33, 1)])
def test_weighted_cov_tensor_cores(n, T, S, NP, cuda):
    """sum_s w_s (x_s - mu)(x_s - mu)^T on tcgen05 (3xTF32) against numpy fp64 and the fp64 CUDA-core kernel.  No reference
    counterpart (diagnostic); full tiles (M = 896), two-tile, and ragged M / S (M = 140, 42; S = 40, 33)."""
    rs = np.random.RandomState(n * 100 + T)
    d = 2 * n
    M = T * d
    mu = rs.normal(0, 1.0, (1, NP, T, d))
    x = mu[..., None] + rs.normal(0, 0.3, (1, NP, T, d, S)) * rs.uniform(0.2, 2.0, (1, NP, T, d, 1))
    w = rs.dirichlet(np.ones(S) * 0.3, (1, NP))
    Y = (x - mu[..., None]).reshape(NP, M, S)
    want = np.einsum('pis,ps,pjs->pij', Y, w[0], Y)
    sh = _ops().make_shape(1, NP, 1, S, T, n, torch.float32)
    xs, mt, wt = (torch.tensor(a, device=cuda, dtype=torch.float32) for a in (x, mu, w))
    Yf = (xs.double() - mt.double().unsqueeze(-1)).reshape(NP, M, S).cpu().numpy()         # the fp32 inputs, exactly
    want32 = np.einsum('pis,ps,pjs->pij', Yf, wt.double().cpu().numpy()[0], Yf)
    got = _ops().weighted_cov(sh, xs, mt, wt, tensor_cores=True).cpu().numpy()[0]
    assert got.shape == (NP, M, M)
    assert rel(got, want32) < 1e-5                   # 3xTF32 + tensor-core fp32 accumulation: 5e-6 measured (plain TF32: ~5e-4)
    assert rel(got, np.transpose(got, (0, 2, 1))) < 1e-5
    simple = _ops().weighted_cov(sh, xs, mt, wt, tensor_cores=False).cpu().numpy()[0]
    assert rel(simple, want32) < 1e-6
    sh64 = _ops().make_shape(1, NP, 1, S, T, n, torch.float64)
    got64 = _ops().weighted_cov(sh64, xs.double(), mt.double(), wt.double()).cpu().numpy()[0]
    assert rel(got64, want32) < 1e-13
    assert rel(want32, want) < 1e-5


def test_planner_weighted_covariance(cuda):
    g = load('panda_soft_f32')
    spec = OP.spec_from_golden(g)
    from stoch_gpmp_b200.planner import StochGPMP
    ta = dict(device=cuda, dtype=torch.float32)
    comp, _ = _lowered(spec, cuda, torch.float32)
    pl = StochGPMP(num_particles_per_goal=spec['K'], num_samples=spec['S'], traj_len=spec['T'], opt_iters=1, dt=spec['dt'], n_dof=spec['n_dof'],
                   step_size=spec['step_size'], temperature=spec['temperature'], start_state=torch.tensor(spec['start'], **ta),
                   multi_goal_states=torch.tensor(spec['goals'], **ta), initial_particle_means='const_vel', cost=comp, seed=3, tensor_args=ta,
                   **{k: spec[k] for k in ('sigma_start_init', 'sigma_gp_init', 'sigma_goal_init', 'sigma_start_sample', 'sigma_gp_sample', 'sigma_goal_sample')})
    pm, vm, ps, vs, costs, grad = pl.optimize(return_samples=True, **_obs(spec, cuda, torch.float32))
    cov = pl.weighted_covariance().cpu().numpy().astype(np.float64)
    x = torch.cat([ps, vs], -1).double().cpu().numpy()                         # [NP,S,T,d]
    mu = torch.cat([pm, vm], -1).double().cpu().numpy()                        # [NP,T,d] (pre-update means)
    w = pl._weights.reshape(pl.num_particles, -1).double().cpu().numpy()
    Y = (x - mu[:, None]).reshape(x.shape[0], x.shape[1], -1)
    want = np.einsum('psi,ps,psj->pij', Y, w, Y)
    assert rel(cov, want) < 2e-5


@pytest.mark.parametrize("n,T,S,NP", [(7, 64, 512, 2), (2, 64, 256, 3), (3, 10, 40, 2), (2, 100, 130, 1)])
def test_sample_dense_tensor_cores_equals_banded(n, T, S, NP, cuda):
    """The dense-L sampling variant (x = mu + L eps as a per-DoF GEMM on tcgen05, 3xTF32) against the banded recurrence of K2
    on the same eps: full tile (2T = 128), ragged S, T not filling a tile, and two row tiles (2T = 200)."""
    rs = np.random.RandomState(n + T)
    spec = dict(T=T, dt=0.05, goals=np.zeros((1, 2 * n)), sigma_start_sample=0.5, sigma_gp_sample=0.8, sigma_goal_sample=0.5)
    tab = _tables(spec, cuda)
    sh = _ops().make_shape(1, NP, 1, S, T, n, torch.float32)
    mu = torch.tensor(rs.normal(0, 1, (1, NP, T, 2 * n)), device=cuda, dtype=torch.float32)
    eps = torch.tensor(rs.normal(0, 1, (1, NP, T, 2 * n, S)), device=cuda, dtype=torch.float32)
    banded = _ops().sample(sh, tab, mu, eps_in=eps)
    dense = _ops().sample_dense_tc(sh, tab, mu, eps)
    y_b = (banded - mu.unsqueeze(-1)).double()
    y_d = (dense - mu.unsqueeze(-1)).double()
    assert float((y_b - y_d).abs().max() / y_b.abs().max()) < 1e-5


# ------------------------------------------------------------------------------------ low-latency iteration
@pytest.mark.parametrize("name", ["panda_soft_f32", "panda_self_f32", "panda_shipped_f32", "planar_soft_f32", "planar_soft_f64", "panda_ee_soft_f64",
                                  "panda_interp_f64", "panda_sdf_f64"])
def test_lowlat_iteration_equals_separate_kernels(name, cuda):
    """sgpmp_iterate_lowlat (few problems: K2 -> cost with thread per (sample, time slice) -> K4 with row chunks, n_iters per call)
    against K2 -> K3 -> K4: identical samples, costs equal up to the rounding of the per-step sum, and the update reproduced by K4
    fed the low-latency path's own costs (the softmax amplifies cost rounding, as in the cluster-mode test)."""
    g = load(name)
    spec = OP.spec_from_golden(g)
    f32 = spec['dtype'] == 'float32'
    dt = torch.float32 if f32 else torch.float64
    tab = _tables(spec, cuda)
    _, low = _lowered(spec, cuda, dt)
    sh = _ops().make_shape(1, spec['G'], spec['K'], spec['S'], spec['T'], spec['n_dof'], dt)
    sp = torch.tensor(spec['spheres'], device=cuda, dtype=dt).unsqueeze(0) if 'spheres' in spec else None
    desc = low.desc(spec['temperature'], sp)
    pre = 'sameL_' if f32 else ''
    mu = torch.tensor(g[pre + 'it0_means_pre'][None], device=cuda)
    for it in range(2):
        xs = _ops().sample(sh, tab, mu, seed=11, draw=it)
        c = _ops().cost(sh, desc, tab, xs, mu)
        mu_l = mu.clone()
        out = _ops().iterate(sh, desc, tab, spec['step_size'], 1, mu_l, seed=11, draw0=it, want_samples=True, lowlat=True)
        assert torch.equal(out['means_pre'], mu)
        assert torch.equal(out['samples'], xs)
        assert float((out['costs'] - c).abs().max() / c.abs().max()) < (4e-6 if f32 else 1e-13)    # two summation orders of the same terms
        mu_k = mu.clone()
        grad, w = _ops().update(sh, spec['temperature'], spec['step_size'], out['costs'], xs, mu_k)
        assert torch.equal(out['weights'], w)
        assert float((out['grad'] - grad).abs().max() / max(float(grad.abs().max()), 1e-30)) < (1e-5 if f32 else 1e-12)
        assert float((mu_l - mu_k).abs().max() / mu_k.abs().max()) < (1e-6 if f32 else 1e-13)
        mu = mu_l
    # two iterations in ONE call == two calls
    mu_2 = torch.tensor(g[pre + 'it0_means_pre'][None], device=cuda)
    _ops().iterate(sh, desc, tab, spec['step_size'], 2, mu_2, seed=11, draw0=0, lowlat=True)
    assert torch.equal(mu_2, mu)


def test_lowlat_dependent_launch_chain_equals_serial_launches(cuda, tmp_path):
    """The low-latency iteration chains its three kernels by programmatic dependent launch (each may start while its predecessor
    drains and waits — griddepcontrol.wait — before its first dependent access).  $SGPMP_PDL is read once per process, so the two
    forms run in two subprocesses: 60 iterations of one Panda problem and of the shipped fp64 planar problem must give bit-identical
    means and costs (a missing wait would show up as a race between iterations)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = r'''
import sys, torch
sys.path.insert(0, %r)
import bench
dev = torch.device("cuda:0")
out = {}
for name in ("panda", "planar_shipped"):
    w = bench.workload(name, 1)
    pl = bench.build_planner(w, 1, dev)
    obs = {"obstacle_spheres": torch.tensor(w["spheres"], dtype=torch.float32, device=dev)} if w["spheres"] is not None else {}
    for rep in range(3):
        r = pl.optimize(opt_iters=20, return_samples=False, **obs)
    out[name + "_means"] = pl._means.cpu()
    out[name + "_costs"] = r[4].cpu()
torch.save(out, sys.argv[1])
''' % root
    res = []
    for flag in ("0", "1"):
        f = str(tmp_path / ("pdl%s.pt" % flag))
        env = dict(os.environ, SGPMP_PDL=flag, SGPMP_LOWLAT="1")
        subprocess.run([sys.executable, "-c", script, f], check=True, env=env, timeout=300)
        res.append(torch.load(f))
    for k in res[0]:
        assert torch.equal(res[0][k], res[1][k]), k
