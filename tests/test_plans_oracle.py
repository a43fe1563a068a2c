"""CPU: the plan oracle's interpolation between support states (oracle/plans.py) against two independent references, and its
selection rule."""
import numpy as np
from scipy.interpolate import CubicHermiteSpline

from oracle import plans as OPL


def _pairs(n=200, seed=0):
    rs = np.random.RandomState(seed)
    return rs.normal(size=(n, 2)), rs.normal(size=(n, 2))


def test_interpolation_is_cubic_hermite():
    dt = 0.05
    xa, xb = _pairs()
    for m in (1, 3, 8, 32):
        lam, psi = OPL.interp_blocks(dt, m)
        for k in range(1, m + 1):
            tau = k * dt / (m + 1)
            x = OPL.interpolate(xa, xb, lam[k - 1], psi[k - 1])
            for a, b, got in zip(xa, xb, x):
                sp = CubicHermiteSpline([0.0, dt], [a[0], b[0]], [a[1], b[1]])
                want = np.array([sp(tau), sp(tau, 1)])
                assert np.abs(got - want).max() <= 1e-11 * max(np.abs(want).max(), 1.0)


def test_interpolation_is_the_gp_conditional_mean():
    """Dense conditional mean of x(tau) given (x_i, x_{i+1}) under the constant-velocity GP (white-noise acceleration, Q_c = 3.7):
    joint Gaussian of [x_i, x(tau), x_{i+1}] with x_i ~ N(0, I), x(tau) = Phi(tau) x_i + w1, x_{i+1} = Phi(dt - tau) x(tau) + w2."""
    dt, qc = 0.05, 3.7
    phi = lambda s: np.array([[1.0, s], [0.0, 1.0]])
    Q = lambda s: qc * np.array([[s ** 3 / 3, s ** 2 / 2], [s ** 2 / 2, s]])
    xa, xb = _pairs(seed=1)
    for m in (1, 4, 9):
        lam, psi = OPL.interp_blocks(dt, m)
        for k in range(1, m + 1):
            tau = k * dt / (m + 1)
            A = np.zeros((6, 6))                 # [x_i; x_tau; x_{i+1}] = A [x_i; w1; w2]
            A[0:2, 0:2] = np.eye(2)
            A[2:4, 0:2], A[2:4, 2:4] = phi(tau), np.eye(2)
            A[4:6, 0:2], A[4:6, 2:4], A[4:6, 4:6] = phi(dt), phi(dt - tau), np.eye(2)
            S0 = np.zeros((6, 6))
            S0[0:2, 0:2], S0[2:4, 2:4], S0[4:6, 4:6] = np.eye(2), Q(tau), Q(dt - tau)
            S = A @ S0 @ A.T
            obs = [0, 1, 4, 5]
            gain = S[np.ix_([2, 3], obs)] @ np.linalg.inv(S[np.ix_(obs, obs)])
            want = (gain @ np.concatenate([xa, xb], axis=1).T).T
            got = OPL.interpolate(xa, xb, lam[k - 1], psi[k - 1])
            assert np.abs(got - want).max() <= 1e-10 * max(np.abs(want).max(), 1.0)


def test_support_states_are_unchanged():
    rs = np.random.RandomState(2)
    means = rs.normal(size=(3, 4, 16, 14))
    for m in (0, 1, 8):
        x = OPL.dense(means, 0.05, m)
        assert x.shape == (3, 4, 15 * (m + 1) + 1, 14)
        assert np.array_equal(x[..., ::m + 1, :], means)


def test_selection_rule():
    inf, nan = np.inf, np.nan
    costs = np.array([[1.0, 2.0, 3.0],        # lowest cost collides -> 1
                      [5.0, 4.0, 4.0],        # tie -> lowest index
                      [3.0, 1.0, 2.0],        # none feasible -> argmin over all
                      [nan, 2.0, 1.0],        # NaN never feasible; 2 collides -> 1
                      [nan, inf, nan]])       # none feasible: +inf ranks before NaN
    clear = np.array([[-0.1, 0.2, 0.3], [0.1, 0.1, 0.1], [-1.0, -1.0, -1.0], [0.5, 0.5, 0.5], [1.0, 1.0, 1.0]])
    hits = np.array([[0, 0, 0], [0, 0, 0], [0, 0, 0], [0, 0, 2], [0, 0, 0]])
    particle, ok = OPL.select(costs, clear, hits, 0.0)
    assert particle.tolist() == [1, 1, 1, 1, 1]
    assert ok.tolist() == [True, True, False, True, False]
