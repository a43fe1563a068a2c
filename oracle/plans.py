"""Oracle: final-plan selection (StochGPMPBatch.best_plans / sgpmp_select_plans), numpy fp64.

TEST INFRASTRUCTURE (see oracle/__init__.py).  No reference counterpart: the reference stops at the particle means.

States between two support states are the constant-velocity GP prior's interpolation, per DoF on (q, qdot):
    x(tau) = Lambda(tau) x_i + Psi(tau) x_{i+1},  Psi = Q(tau) Phi(dt - tau)^T Q(dt)^-1,  Lambda = Phi(tau) - Psi Phi(dt)
with Phi(s) = [[1, s], [0, 1]] and Q(s) = [[s^3/3, s^2/2], [s^2/2, s]] (the power-spectral density Q_c cancels).  A mean of T
support states is checked at P = (T-1)(m+1)+1 states: state j lies in interval i = j // (m+1) at tau = (j % (m+1)) dt / (m+1).
"""
import numpy as np

from . import costs as _costs
from . import fk as _fk


def _phi(s):
    return np.array([[1.0, s], [0.0, 1.0]])


def _q(s):
    return np.array([[s ** 3 / 3, s ** 2 / 2], [s ** 2 / 2, s]])


def interp_blocks(dt, m):
    """(Lambda [m,2,2], Psi [m,2,2]) for tau_k = k dt / (m+1), k = 1..m."""
    lam, psi = [], []
    qinv = np.linalg.inv(_q(dt))
    for k in range(1, m + 1):
        tau = k * dt / (m + 1)
        ps = _q(tau) @ _phi(dt - tau).T @ qinv
        lam.append(_phi(tau) - ps @ _phi(dt))
        psi.append(ps)
    return np.array(lam).reshape(m, 2, 2), np.array(psi).reshape(m, 2, 2)


def interpolate(xa, xb, lam, psi):
    """x(tau) of one interval: xa, xb [..., d] = [q(n), qdot(n)]; lam, psi [2,2] -> [..., d]."""
    n = xa.shape[-1] // 2
    qa, va, qb, vb = xa[..., :n], xa[..., n:], xb[..., :n], xb[..., n:]
    q = lam[0, 0] * qa + lam[0, 1] * va + psi[0, 0] * qb + psi[0, 1] * vb
    v = lam[1, 0] * qa + lam[1, 1] * va + psi[1, 0] * qb + psi[1, 1] * vb
    return np.concatenate([q, v], axis=-1)


def dense(means, dt, m):
    """means [..., T, d] -> [..., P, d]; every (m+1)-th state is the support state itself, unchanged."""
    means = np.asarray(means, dtype=np.float64)
    T, d = means.shape[-2], means.shape[-1]
    lam, psi = interp_blocks(dt, m)
    out = np.empty(means.shape[:-2] + ((T - 1) * (m + 1) + 1, d))
    out[..., ::m + 1, :] = means
    for k in range(1, m + 1):
        out[..., k::m + 1, :] = interpolate(means[..., :-1, :], means[..., 1:, :], lam[k - 1], psi[k - 1])
    return out


def clearance(means, spheres, dt, m, num_interpolate=0, interp_range=(5, 7), include_base=True):
    """Least |p - c| - r over the checked states t > 0 of every mean [..., T, d] (Panda chain), the sphere field's points (link
    origins + link interpolation) and the spheres [O, 4] -> [...]."""
    x = dense(means, dt, m)[..., 1:, :]
    n = x.shape[-1] // 2
    H = _fk.fk_all_links(x[..., :n].reshape(-1, n), include_base=include_base)
    pos = _costs.interpolate_links(H[:, :, :3, 3], num_interpolate, interp_range)          # [N, L', 3]
    sp = np.asarray(spheres, dtype=np.float64)
    dist = np.linalg.norm(pos[:, :, None, :] - sp[None, None, :, :3], axis=-1) - sp[:, 3]
    return dist.reshape(x.shape[:-1] + (-1,)).min(axis=(-1, -2))


def hits(means, occ_map, cell_size, origin_xi, origin_yi, dt, m):
    """Number of checked states t > 0 of every mean [..., T, d] whose occupancy cell is non-zero -> [...]."""
    x = dense(means, dt, m)[..., 1:, :2]
    return (_costs.map_lookup(x, occ_map, cell_size, origin_xi, origin_yi) != 0).sum(-1)


def select(costs, clearance_, hits_, margin):
    """Per problem (rows): argmin cost over the feasible particles (no hit, clearance >= margin, finite cost), ties to the lowest
    index; with none feasible, argmin over all with NaN last.  -> (particle [B], ok [B] bool)."""
    costs = np.asarray(costs)
    feas = (np.asarray(hits_) == 0) & (np.asarray(clearance_) >= margin) & np.isfinite(costs)
    particle, ok = [], []
    for c, f in zip(costs, feas):
        pool = np.flatnonzero(f) if f.any() else np.arange(len(c))
        particle.append(min(pool, key=lambda p: (bool(np.isnan(c[p])), 0.0 if np.isnan(c[p]) else float(c[p]), int(p))))
        ok.append(bool(f.any()))
    return np.array(particle), np.array(ok)
