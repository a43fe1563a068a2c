"""CPU: the C-ABI library loads and exports every symbol include/stoch_gpmp_b200.h declares; host-side
logic (cost lowering, map generation, error behaviour) without any compute call."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    txt = open(os.path.join(ROOT, "include", "stoch_gpmp_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(sgpmp_[a-z_A-Z0-9]+)\s*\(", txt)))


def test_header_symbols_exported(lib):
    from stoch_gpmp_b200 import _lib
    syms = _declared_symbols()
    assert len(syms) >= 12
    raw = ctypes.CDLL(_lib.lib_path())
    for s in syms:
        assert hasattr(raw, s), "library does not export %s" % s
    assert set(syms) == set(_lib.SIGNATURES), "ctypes binding and header disagree"
    assert lib.sgpmp_abi_version() == _lib.ABI_VERSION


def test_struct_layout_matches_c(lib, tmp_path):
    """sizeof/offsetof of the two POD structs as gcc sees them == the ctypes mirrors."""
    from stoch_gpmp_b200 import _lib
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "stoch_gpmp_b200.h"\nint main(){'
                   'printf("%zu %zu %zu %zu %zu %zu %zu\\n", sizeof(sgpmp_shape_t), sizeof(sgpmp_cost_desc_t),'
                   'offsetof(sgpmp_cost_desc_t, start), offsetof(sgpmp_cost_desc_t, map_inv_cell),'
                   'offsetof(sgpmp_cost_desc_t, spheres), offsetof(sgpmp_cost_desc_t, chain_R),'
                   'offsetof(sgpmp_cost_desc_t, chain_joint));return 0;}')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    D = _lib.CostDesc
    want = [ctypes.sizeof(_lib.Shape), ctypes.sizeof(D), D.start.offset, D.map_inv_cell.offset, D.spheres.offset,
            D.chain_R.offset, D.chain_joint.offset]
    assert got == want


def test_dof_support_table(lib):
    assert lib.sgpmp_dof_supported(2) == 1 and lib.sgpmp_dof_supported(7) == 1
    assert lib.sgpmp_dof_supported(5) == 1 and lib.sgpmp_dof_supported(14) == 1      # every DoF count of BASELINE's C5 sweep
    assert lib.sgpmp_dof_supported(9) == 0 and lib.sgpmp_dof_supported(0) == 0


def test_bad_arguments_are_reported_not_crashed(lib):
    from stoch_gpmp_b200 import _lib
    rc = lib.sgpmp_prior_factor(0, 1, None, None, None, None, None)
    assert rc == _lib.ERR_INVALID_ARG and b"T >= 2" in lib.sgpmp_last_error()
    sh = _lib.Shape(B=1, G=1, K=1, S=1, T=1, n_dof=2, dtype=0)
    assert lib.sgpmp_sample(ctypes.byref(sh), None, None, None, 0, 0, None, None, None) == _lib.ERR_INVALID_ARG
    with pytest.raises(ValueError):
        _lib.check(_lib.ERR_INVALID_ARG, "x")
    with pytest.raises(NotImplementedError):
        _lib.check(_lib.ERR_UNSUPPORTED, "x")


def test_no_cpu_fallback():
    from stoch_gpmp_b200 import ops
    from stoch_gpmp_b200.planner import StochGPMP
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.prior_factor(torch.zeros(1, 4, 3, dtype=torch.float64), torch.zeros(1, 3, 4, dtype=torch.float64))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        StochGPMP(1, 4, 8, 1, dt=0.1, n_dof=2, start_state=torch.zeros(4), multi_goal_states=torch.zeros(1, 4),
                  tensor_args={'device': torch.device('cpu'), 'dtype': torch.float32})


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from stoch_gpmp_b200 import _lib, build
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(build, "LIB", str(tmp_path / "nope.so"))
    with pytest.raises(ImportError, match="no CPU fallback"):
        _lib.load()


def test_product_does_not_import_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference arm may touch oracle/."""
    pkg = os.path.join(ROOT, "stoch_gpmp_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".inc")):
                txt = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f
                assert "/root/reference" not in txt or f.endswith((".cu", ".cuh", ".py")) and "import" not in txt.split("/root/reference")[0][-20:], f
    code = "import sys; import stoch_gpmp_b200.planner, stoch_gpmp_b200.costs.cost_functions, stoch_gpmp_b200.envs.map_generator; " \
           "assert not any(m == 'oracle' or m.startswith('oracle.') for m in sys.modules), 'oracle imported'"
    subprocess.check_call([sys.executable, "-c", code], cwd=ROOT)


def test_prior_blocks_equal_oracle():
    from oracle import prior as P
    from stoch_gpmp_b200.planner import prior_blocks
    for (T, dt, ss, sg, sgo) in [(16, 0.02, 1e-3, 3.0, 1e-3), (64, 0.05, 1e-4, 0.8, 0.1), (9, 0.1, 0.5, 2.0, None)]:
        D, O = prior_blocks(T, dt, ss, sg, sgo)
        D2, O2 = P.precision_blocks(T, dt, ss, sg, sgo)
        assert np.array_equal(np.array(D), np.stack([D2[:, 0, 0], D2[:, 0, 1], D2[:, 1, 1]], 1))
        assert np.array_equal(np.array(O), O2.reshape(-1, 4))


def test_generate_obstacle_map_matches_golden_map():
    """Same seeds -> the same occupancy grid as the reference's generator (golden 'map' arrays)."""
    import random
    from stoch_gpmp_b200.envs.map_generator import generate_obstacle_map
    from helpers import load
    ta = {'device': torch.device('cpu'), 'dtype': torch.float64}
    random.seed(0)
    np.random.seed(0)
    m = generate_obstacle_map(map_dim=[20, 20], obst_list=[], cell_size=0.1, random_gen=True, num_obst=15,
                              rand_limits=[[-7.5, 7.5], [-7.5, 7.5]], rand_rect_shape=[2, 2], tensor_args=ta)[0]
    assert np.array_equal(m.map, load('planar_f64')['map'])
    assert (m.origin_xi, m.origin_yi) == tuple(load('planar_f64')['map_origin'])
    random.seed(1)
    np.random.seed(1)
    m = generate_obstacle_map(map_dim=[8, 8], obst_list=[], cell_size=0.1, random_gen=True, num_obst=4,
                              rand_limits=[[-1.5, 1.5], [-1.5, 1.5]], rand_rect_shape=[2, 2], tensor_args=ta)[0]
    assert np.array_equal(m.map, load('planar_soft_f64')['map'])


def test_cost_lowering_rejects_what_it_cannot_lower():
    from stoch_gpmp_b200.costs.cost_functions import CostCollision, CostComposite, CostGP, CostGoal
    from stoch_gpmp_b200.costs.fields import LinkDistanceField, LinkSelfDistanceField, EESE3DistanceField
    from stoch_gpmp_b200.envs.occupancy import ObstacleMap
    ta = {'device': torch.device('cpu'), 'dtype': torch.float32}
    gp = CostGP(7, 8, torch.zeros(14), 0.05, dict(sigma_start=1., sigma_gp=1.), ta)
    with pytest.raises(NotImplementedError):
        LinkSelfDistanceField(num_interpolate=9).check_lowerable()       # more than SGPMP_MAX_INTERP
    LinkSelfDistanceField(num_interpolate=2).check_lowerable()
    with pytest.raises(NotImplementedError, match="SerialChainFK"):
        CostComposite(7, 8, [gp, CostCollision(7, 8, field=LinkSelfDistanceField(), sigma_coll=1.)], FK=None).lower(
            1, 1, torch.device('cpu'), torch.float32)
    # CostGoal: only the EE SE(3) field lowers; one target pose; FK descriptor required
    with pytest.raises(NotImplementedError, match="CostGoal field"):
        CostComposite(7, 8, [gp, CostGoal(7, 8, field=LinkDistanceField(), sigma_goal=1.)]).lower(1, 1, torch.device('cpu'), torch.float32)
    with pytest.raises(NotImplementedError, match="one target pose"):
        EESE3DistanceField(torch.eye(4).repeat(2, 1, 1)).check_lowerable()
    with pytest.raises(NotImplementedError, match="SerialChainFK"):
        CostComposite(7, 8, [gp, CostGoal(7, 8, field=EESE3DistanceField(torch.eye(4)), sigma_goal=1.)], FK=None).lower(
            1, 1, torch.device('cpu'), torch.float32)
    CostComposite(7, 8, [gp, CostGoal(7, 8)]).lower(1, 1, torch.device('cpu'), torch.float32)    # field=None: term dropped
    # LinkDistanceField under an FK callable that is not a SerialChainFK descriptor: not lowered, kept as a torch-evaluated term
    # (the reference accepts any FK callable, cost_functions.py:39-52; tests/test_gpu_planner.py::test_arbitrary_fk_callable)
    fk_any = lambda q: q
    coll_any = CostCollision(7, 8, field=LinkDistanceField(), sigma_coll=1.)
    low_any = CostComposite(7, 8, [gp, coll_any], FK=fk_any).lower(1, 1, torch.device('cpu'), torch.float32)
    assert low_any.fk is None and low_any.sphere_sigma is None and len(low_any.custom) == 1
    assert low_any.custom[0].__self__ is coll_any
    with pytest.raises(NotImplementedError):
        LinkDistanceField(field_type='hinge').check_lowerable()
    with pytest.raises(NotImplementedError):
        LinkDistanceField(num_interpolate=30).check_lowerable()
    assert LinkDistanceField(num_interpolate=3).interp_alpha() == [0.25, 0.5, 0.75]
    assert LinkDistanceField(field_type='sdf', clamp_sdf=True).field_code() == 2
    # non-square map
    om = ObstacleMap([4, 2], 0.5, tensor_args=ta)
    gp2 = CostGP(2, 8, torch.zeros(4), 0.05, dict(sigma_start=1., sigma_gp=1.), ta)
    with pytest.raises(NotImplementedError, match="non-square"):
        CostComposite(2, 8, [gp2, CostCollision(2, 8, field=om, sigma_coll=1.)]).lower(1, 1, torch.device('cpu'), torch.float32)
    with pytest.raises(NotImplementedError, match="CostGP"):
        CostComposite(2, 8, []).lower(1, 1, torch.device('cpu'), torch.float32)


def test_ee_goal_and_interpolation_reach_the_descriptor():
    from stoch_gpmp_b200.costs.cost_functions import CostCollision, CostComposite, CostGP, CostGoal
    from stoch_gpmp_b200.costs.fields import LinkDistanceField, LinkSelfDistanceField, EESE3DistanceField
    from stoch_gpmp_b200.robots import PandaFK
    ta = {'device': torch.device('cpu'), 'dtype': torch.float64}
    gp = CostGP(7, 8, torch.zeros(14), 0.05, dict(sigma_start=1., sigma_gp=1.), ta)
    H = torch.eye(4, dtype=torch.float64)
    H[:3, 3] = torch.tensor([.3, .2, .1], dtype=torch.float64)
    fld = EESE3DistanceField(H.unsqueeze(0), w_pos=2., w_rot=.5, square=False, tensor_args=ta)
    comp = CostComposite(7, 8, [gp, CostCollision(7, 8, field=LinkSelfDistanceField(num_interpolate=2, link_interpolate_range=[3, 6]), sigma_coll=1.),
                                CostCollision(7, 8, field=LinkDistanceField(num_interpolate=3), sigma_coll=1.),
                                CostGoal(7, 8, field=fld, sigma_goal=0.5)], FK=PandaFK())
    low = comp.lower(1, 1, torch.device('cpu'), torch.float64)
    d = low.desc(1.0, torch.zeros(1, 2, 4, dtype=torch.float64))
    assert (d.self_interp_n, d.self_interp_lo, d.self_interp_hi) == (2, 3, 6)
    assert (d.sphere_interp_n, d.sphere_interp_lo, d.sphere_interp_hi) == (3, 5, 7)
    assert list(d.sphere_interp_alpha)[:3] == [0.25, 0.5, 0.75]
    assert [float(a) for a in torch.linspace(0, 1, 4)[1:3]] == list(d.self_interp_alpha)[:2]      # float32 fractions, fields.py:69
    assert d.ee_sigma_goal == 0.5 and (d.ee_w_pos, d.ee_w_rot, d.ee_square) == (2., .5, 0)
    assert list(d.ee_target_p) == [.3, .2, .1] and list(d.ee_target_R) == [1, 0, 0, 0, 1, 0, 0, 0, 1]
    H2 = H.clone()
    H2[0, 3] = 0.9
    fld.update_target(H2)                                       # fields.py:139-140
    assert low.desc(1.0, torch.zeros(1, 2, 4, dtype=torch.float64)).ee_target_p[0] == 0.9


def test_interp_alpha_and_se3_oracle():
    """oracle.costs.interp_alpha == torch.linspace(0, 1, n+2)[1:n+1] (float32, then cast: costs/fields.py:69);
    oracle.se3: identities of the restated SE3_distance."""
    from oracle.costs import interp_alpha
    from oracle.se3 import se3_distance, se3_distance_torch
    for n in range(1, 17):
        a = torch.linspace(0, 1, n + 2)[1:n + 1]
        assert np.array_equal(a.numpy().astype(np.float64), interp_alpha(n, np.float64))
    H = np.eye(4)
    c, s_ = np.cos(0.7), np.sin(0.7)
    H2 = np.eye(4)
    H2[:3, :3] = [[c, -s_, 0], [s_, c, 0], [0, 0, 1]]
    H2[:3, 3] = [3., 4., 0.]
    assert se3_distance(H, H) == 0.0
    assert abs(se3_distance(H2, H, 2.0, 0.5) - (2.0 * 5.0 + 0.5 * 0.7)) < 1e-12
    assert abs(float(se3_distance_torch(torch.tensor(H2), torch.tensor(H), 2.0, 0.5)) - (10.0 + 0.35)) < 1e-12


def test_panda_chain_from_urdf_equals_builtin():
    """The embedded chain constants == what the reference's URDF says: its joints as stored in tests/golden/ and, where a
    reference checkout is found (oracle/ref_loader.py: $STOCH_GPMP_REF), the original file."""
    from oracle.ref_loader import reference_root
    from stoch_gpmp_b200.robots import PandaFK, SerialChainFK
    urdfs = [os.path.join(ROOT, "tests", "golden", "panda_arm_no_gripper_joints.urdf")]
    if reference_root() is not None:
        urdfs.append(os.path.join(reference_root(), "assets", "franka_description", "robots", "panda_arm_no_gripper.urdf"))
    b = PandaFK()
    for urdf in urdfs:
        a = SerialChainFK.from_urdf(urdf, "panda_link0", "ee_link")
        assert a.names == b.names and a.joint == b.joint and a.xyz == b.xyz, urdf
        assert np.allclose(np.array(a.R), np.array(b.R), atol=0), urdf
    assert b.num_links == 11 and b.n_dofs == 7


def test_merge_stats_is_logsumexp_merge():
    from stoch_gpmp_b200.ops import merge_stats
    rs = np.random.RandomState(0)
    z = torch.tensor(rs.randn(2, 3, 40) * 5)       # [B,NP,S] logits
    eps = torch.tensor(rs.randn(2, 3, 6, 40))      # [B,NP,M,S]

    def stats(sl):
        zz, ee = z[..., sl], eps[..., sl]
        m = zz.max(-1).values
        w = torch.exp(zz - m.unsqueeze(-1))
        return torch.cat([m.unsqueeze(-1), w.sum(-1, keepdim=True), (ee * w.unsqueeze(-2)).sum(-1)], -1)
    merged = merge_stats([stats(slice(0, 13)), stats(slice(13, 40))])
    full = stats(slice(0, 40))
    assert torch.allclose(merged[..., 2:] / merged[..., 1:2], full[..., 2:] / full[..., 1:2], atol=1e-12)
    assert torch.allclose(merged[..., 0], full[..., 0])


def test_serial_chain_fk_callable_matches_oracle_and_custom_terms_are_collected():
    """SerialChainFK.__call__ is the FK hook user-defined cost terms receive x_trajs from (cost_functions.py:51-52 convention):
    all link frames as 4x4 transforms, equal to oracle/fk.py; callables in cost_list are collected as user terms by lower()."""
    from oracle import fk as OFK
    from stoch_gpmp_b200.costs.cost_functions import CostComposite, CostGP
    from stoch_gpmp_b200.robots import PandaFK
    q = np.random.RandomState(3).uniform(-2.5, 2.5, (4, 6, 7))
    H = PandaFK()(torch.tensor(q)).numpy()
    assert H.shape == (4, 6, 11, 4, 4)
    assert np.abs(H - OFK.fk_all_links(q.reshape(-1, 7)).reshape(H.shape)).max() < 1e-14
    assert PandaFK(include_base=False)(torch.tensor(q[0])).shape == (6, 10, 4, 4)
    ta = {'device': torch.device('cpu'), 'dtype': torch.float64}
    gp = CostGP(7, 8, torch.zeros(14), 0.05, dict(sigma_start=1., sigma_gp=1.), ta)

    def term(trajs, x_trajs=None, **obs):
        return x_trajs[:, :, -1, 2, 3].sum(-1) + obs['bias']
    low = CostComposite(7, 8, [gp, term], FK=PandaFK()).lower(1, 1, torch.device('cpu'), torch.float64)
    assert low.custom == [term]
    trajs = torch.tensor(np.random.RandomState(4).randn(5, 8, 14))
    want = PandaFK()(trajs[..., :7])[:, :, -1, 2, 3].sum(-1) + 2.0
    assert torch.allclose(low.custom_costs(trajs, bias=2.0), want)
    with pytest.raises(NotImplementedError, match="not callable"):
        CostComposite(7, 8, [gp, object()]).lower(1, 1, torch.device('cpu'), torch.float64)
