"""Tensor-level wrappers over the C-ABI (include/stoch_gpmp_b200.h).

torch is used for device memory and the current stream only; all arithmetic happens in libsgpmp.so.
Every function raises if handed CPU tensors: there is no CPU path in this package.
"""
import ctypes as C

import torch

from . import _lib

_DT = {torch.float32: _lib.SGPMP_F32, torch.float64: _lib.SGPMP_F64}


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream():
    """cudaStream_t of torch's current stream on the current device (callers sit inside `with torch.cuda.device(...)`).  The raw
    query is ~10x cheaper than torch.cuda.current_stream(); it matters for the reference's usage pattern, a Python loop of
    single-iteration optimize() calls, which is host-bound."""
    if _raw_stream is not None:
        return C.c_void_p(_raw_stream(torch.cuda.current_device()))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class _on_device:
    """`with torch.cuda.device(dev)` costs ~5 us per call; the reference's usage pattern (a Python loop of single-iteration
    optimize() calls) is host-bound, so the switch is skipped when `dev` already is the current device."""
    __slots__ = ("ctx",)

    def __init__(self, dev):
        self.ctx = None if (dev.index is None or dev.index == torch.cuda.current_device()) else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *a):
        if self.ctx is not None:
            self.ctx.__exit__(*a)


def _req(t, name, dtype=None, shape=None):
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor" % name)
    if not t.is_cuda:
        raise RuntimeError("%s is on %s — stoch_gpmp_b200 runs on CUDA devices only (no CPU fallback)" % (name, t.device))
    if dtype is not None and t.dtype != dtype:
        raise TypeError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    if shape is not None and tuple(t.shape) != tuple(shape):
        raise ValueError("%s must have shape %s, got %s" % (name, tuple(shape), tuple(t.shape)))
    return t


def make_shape(B, G, K, S, T, n_dof, dtype, problem_gid0=0, sample_gid0=0):
    if dtype not in _DT:
        raise TypeError("dtype must be torch.float32 or torch.float64, got %s" % dtype)
    return _lib.Shape(B=B, G=G, K=K, S=S, T=T, n_dof=n_dof, dtype=_DT[dtype], sample_gid0=sample_gid0, problem_gid0=problem_gid0)


def prior_factor(D, O):
    """K1.  D [n_priors,T,3], O [n_priors,T-1,4] (float64, CUDA) -> (tables [n_priors,T,16], not_pd [n_priors])."""
    lib = _lib.load()
    _req(D, "D", torch.float64)
    _req(O, "O", torch.float64)
    n, T = D.shape[0], D.shape[1]
    if tuple(D.shape) != (n, T, 3) or tuple(O.shape) != (n, T - 1, 4):
        raise ValueError("prior_factor: D must be [n,T,3] and O [n,T-1,4]")
    tables = torch.empty(n, T, _lib.TABLE_STRIDE, dtype=torch.float64, device=D.device)
    not_pd = torch.empty(n, dtype=torch.int32, device=D.device)
    with torch.cuda.device(D.device):
        _lib.check(lib.sgpmp_prior_factor(n, T, _ptr(D), _ptr(O), _ptr(tables), _ptr(not_pd), _stream()), "sgpmp_prior_factor")
    return tables, not_pd


def prior_dense_L(tables, n_dof, dtype):
    """Dense scale_tril [M,M] of one prior (tables [T,16])."""
    lib = _lib.load()
    _req(tables, "tables", torch.float64)
    T = tables.shape[0]
    M = T * 2 * n_dof
    L = torch.empty(M, M, dtype=dtype, device=tables.device)
    with torch.cuda.device(tables.device):
        _lib.check(lib.sgpmp_prior_dense_L(T, n_dof, _ptr(tables), _DT[dtype], _ptr(L), _stream()), "sgpmp_prior_dense_L")
    return L


def sample(shape, tables, means, eps_in=None, seed=0, draw=0, want_eps=False):
    """K2.  means [B,NP,T,d] -> samples [B,NP,T,d,S] (S-minor).  eps_in, if given, has the samples layout."""
    lib = _lib.load()
    B, NP, T, d, S = shape.B, shape.G * shape.K, shape.T, 2 * shape.n_dof, shape.S
    dt = means.dtype
    _req(tables, "tables", torch.float64, (T, _lib.TABLE_STRIDE))
    _req(means, "means", None, (B, NP, T, d))
    if eps_in is not None:
        _req(eps_in, "eps_in", dt, (B, NP, T, d, S))
    out = torch.empty(B, NP, T, d, S, dtype=dt, device=means.device)
    eps_out = torch.empty_like(out) if want_eps else None
    with torch.cuda.device(means.device):
        _lib.check(lib.sgpmp_sample(C.byref(shape), _ptr(tables), _ptr(means), _ptr(eps_in), seed, draw, _ptr(out),
                                    _ptr(eps_out), _stream()), "sgpmp_sample")
    return (out, eps_out) if want_eps else out


def cost(shape, desc, tables, samples, means=None, want_terms=False):
    """K3.  samples [B,NP,T,d,S] -> costs [B,NP,S] (+ terms [5,B,NP,S]).  means=None drops the IS term."""
    lib = _lib.load()
    B, NP, T, d, S = shape.B, shape.G * shape.K, shape.T, 2 * shape.n_dof, shape.S
    dt = samples.dtype
    _req(samples, "samples", None, (B, NP, T, d, S))
    if means is not None:
        _req(tables, "tables", torch.float64, (T, _lib.TABLE_STRIDE))
        _req(means, "means", dt, (B, NP, T, d))
    costs = torch.empty(B, NP, S, dtype=dt, device=samples.device)
    terms = torch.empty(_lib.NUM_TERMS, B, NP, S, dtype=dt, device=samples.device) if want_terms else None
    with torch.cuda.device(samples.device):
        _lib.check(lib.sgpmp_cost(C.byref(shape), C.byref(desc), _ptr(tables), _ptr(samples), _ptr(means), _ptr(costs),
                                  _ptr(terms), _stream()), "sgpmp_cost")
    return (costs, terms) if want_terms else costs


def update(shape, temperature, step_size, costs, samples, means):
    """K4.  Updates `means` in place; returns (grad [B,NP,T,d], weights [B,NP,S])."""
    lib = _lib.load()
    B, NP, T, d, S = shape.B, shape.G * shape.K, shape.T, 2 * shape.n_dof, shape.S
    dt = means.dtype
    _req(costs, "costs", dt, (B, NP, S))
    _req(samples, "samples", dt, (B, NP, T, d, S))
    _req(means, "means", None, (B, NP, T, d))
    grad = torch.empty_like(means)
    weights = torch.empty_like(costs)
    with torch.cuda.device(means.device):
        _lib.check(lib.sgpmp_update(C.byref(shape), float(temperature), float(step_size), _ptr(costs), _ptr(samples),
                                    _ptr(means), _ptr(grad), _ptr(weights), _stream()), "sgpmp_update")
    return grad, weights


def iterate(shape, desc, tables, step_size, n_iters, means, eps_in=None, seed=0, draw0=0,
            want_samples=False, want_costs=True, want_weights=True, want_grad=True, want_means_pre=True, lowlat=False,
            validate=True):
    """Fused loop.  Updates `means` in place.  Returns dict(means_pre, samples, costs, weights, grad) of the
    LAST iteration (entries not requested are None).  validate=False skips the argument checks (the planner passes its
    own tensors; the checks are ~2 us of a host-bound call)."""
    lib = _lib.load()
    B, NP, T, d, S = shape.B, shape.G * shape.K, shape.T, 2 * shape.n_dof, shape.S
    dt, dev = means.dtype, means.device
    if validate:
        _req(tables, "tables", torch.float64, (T, _lib.TABLE_STRIDE))
        _req(means, "means", None, (B, NP, T, d))
        if eps_in is not None:
            _req(eps_in, "eps_in", dt, (n_iters, B, NP, T, d, S))
    if lowlat:
        # few problems: three short launches per iteration instead of the thread-per-sample fused kernel (csrc/sgpmp_lowlat.cu)
        out = dict(means_pre=torch.empty_like(means) if want_means_pre else None,
                   samples=torch.empty(B, NP, T, d, S, dtype=dt, device=dev),
                   costs=torch.empty(B, NP, S, dtype=dt, device=dev),
                   weights=torch.empty(B, NP, S, dtype=dt, device=dev) if want_weights else None,
                   grad=torch.empty_like(means) if want_grad else None)
        with _on_device(dev):
            _lib.check(lib.sgpmp_iterate_lowlat(C.byref(shape), C.byref(desc), _ptr(tables), float(step_size), int(n_iters),
                                                _ptr(eps_in), seed, draw0, _ptr(means), _ptr(out["means_pre"]), _ptr(out["samples"]),
                                                _ptr(out["costs"]), _ptr(out["weights"]), _ptr(out["grad"]), _stream()),
                       "sgpmp_iterate_lowlat")
        if not want_samples:
            out["samples"] = None
        return out
    out = dict(
        means_pre=torch.empty_like(means) if want_means_pre else None,
        samples=torch.empty(B, NP, T, d, S, dtype=dt, device=dev) if want_samples else None,
        costs=torch.empty(B, NP, S, dtype=dt, device=dev) if want_costs else None,
        weights=torch.empty(B, NP, S, dtype=dt, device=dev) if want_weights else None,
        grad=torch.empty_like(means) if want_grad else None,
    )
    with _on_device(dev):
        _lib.check(lib.sgpmp_iterate(C.byref(shape), C.byref(desc), _ptr(tables), float(step_size), int(n_iters),
                                     _ptr(eps_in), seed, draw0, _ptr(means), _ptr(out["means_pre"]), _ptr(out["samples"]),
                                     _ptr(out["costs"]), _ptr(out["weights"]), _ptr(out["grad"]), _stream()),
                   "sgpmp_iterate")
    return out


def local_stats(shape, temperature, costs, eps):
    """Split-particle mode: (m, Z, A[M]) per particle of this rank's samples -> stats [B,NP,M+2]."""
    lib = _lib.load()
    B, NP, T, d, S = shape.B, shape.G * shape.K, shape.T, 2 * shape.n_dof, shape.S
    dt = costs.dtype
    _req(costs, "costs", None, (B, NP, S))
    _req(eps, "eps", dt, (B, NP, T, d, S))
    stats = torch.empty(B, NP, T * d + 2, dtype=dt, device=costs.device)
    with torch.cuda.device(costs.device):
        _lib.check(lib.sgpmp_local_stats(C.byref(shape), float(temperature), _ptr(costs), _ptr(eps), _ptr(stats), _stream()),
                   "sgpmp_local_stats")
    return stats


def apply_stats(shape, tables, step_size, stats, means):
    """mu += step * L (A/Z) in place; returns grad."""
    lib = _lib.load()
    B, NP, T, d = shape.B, shape.G * shape.K, shape.T, 2 * shape.n_dof
    _req(stats, "stats", means.dtype, (B, NP, T * d + 2))
    _req(means, "means", None, (B, NP, T, d))
    grad = torch.empty_like(means)
    with torch.cuda.device(means.device):
        _lib.check(lib.sgpmp_apply_stats(C.byref(shape), _ptr(tables), float(step_size), _ptr(stats), _ptr(means), _ptr(grad),
                                         _stream()), "sgpmp_apply_stats")
    return grad


def iterate_stats(shape, desc, tables, means, seed, draw, want_costs=False):
    """Split-particle mode, one fused launch: sample -> cost -> local softmax statistics over the samples
    [shape.sample_gid0, + shape.S) of every particle.  Returns (stats [B,NP,M+2] = (m, Z, A), costs [B,NP,S] or None)."""
    lib = _lib.load()
    B, NP, T, d, S = shape.B, shape.G * shape.K, shape.T, 2 * shape.n_dof, shape.S
    _req(means, "means", None, (B, NP, T, d))
    stats = torch.empty(B, NP, T * d + 2, dtype=means.dtype, device=means.device)
    costs = torch.empty(B, NP, S, dtype=means.dtype, device=means.device) if want_costs else None
    with torch.cuda.device(means.device):
        _lib.check(lib.sgpmp_iterate_stats(C.byref(shape), C.byref(desc), _ptr(tables), int(seed) & (2 ** 64 - 1), int(draw),
                                           _ptr(means), _ptr(costs), _ptr(stats), _stream()), "sgpmp_iterate_stats")
    return stats, costs


def merge_apply_stats(shape, tables, step_size, stats_all, means):
    """stats_all [R,B,NP,M+2] (rank-major) -> in-kernel log-sum-exp merge -> mu += step * L (A/Z) in place; returns grad."""
    lib = _lib.load()
    B, NP, T, d = shape.B, shape.G * shape.K, shape.T, 2 * shape.n_dof
    if stats_all.dim() == 3:
        stats_all = stats_all.unsqueeze(0)
    R = stats_all.shape[0]
    _req(stats_all, "stats_all", means.dtype, (R, B, NP, T * d + 2))
    _req(means, "means", None, (B, NP, T, d))
    grad = torch.empty_like(means)
    with torch.cuda.device(means.device):
        _lib.check(lib.sgpmp_merge_apply_stats(C.byref(shape), _ptr(tables), float(step_size), _ptr(stats_all), int(R), _ptr(means),
                                               _ptr(grad), _stream()), "sgpmp_merge_apply_stats")
    return grad


def iterate_split_particles(shape_local, desc, tables, step_size, n_iters, means, seed, draw0, comm=None, n_ranks=1,
                            want_costs=True, want_grad=True, want_means_pre=True):
    """n_iters split-particle iterations enqueued by ONE C call: per iteration a fused stats launch over this rank's samples,
    one ncclAllGather on the same stream (comm = parallel.NcclComm handle; None iff n_ranks == 1) and one merge + update launch.
    `means` is updated in place (identically on every rank).  Returns dict(means_pre, costs (local), grad)."""
    lib = _lib.load()
    B, NP, T, d, S = shape_local.B, shape_local.G * shape_local.K, shape_local.T, 2 * shape_local.n_dof, shape_local.S
    _req(means, "means", None, (B, NP, T, d))
    dt, dev = means.dtype, means.device
    stats_local = torch.empty(B, NP, T * d + 2, dtype=dt, device=dev)
    stats_all = torch.empty(n_ranks, B, NP, T * d + 2, dtype=dt, device=dev) if n_ranks > 1 else None
    out = dict(means_pre=torch.empty_like(means) if want_means_pre else None,
               costs=torch.empty(B, NP, S, dtype=dt, device=dev) if want_costs else None,
               grad=torch.empty_like(means) if want_grad else None)
    with torch.cuda.device(dev):
        _lib.check(lib.sgpmp_iterate_split_particles(C.byref(shape_local), C.byref(desc), _ptr(tables), float(step_size), int(n_iters),
                                                     int(seed) & (2 ** 64 - 1), int(draw0), _ptr(means), _ptr(out["means_pre"]),
                                                     C.c_void_p(comm) if comm else None, int(n_ranks), _ptr(stats_local), _ptr(stats_all),
                                                     _ptr(out["costs"]), _ptr(out["grad"]), _stream()), "sgpmp_iterate_split_particles")
    out["_keepalive"] = (stats_local, stats_all)      # the launches are asynchronous: keep the exchange buffers until the caller is done
    return out


def merge_stats(stats_list):
    """Log-sum-exp merge of per-rank (m, Z, A) statistics (the arithmetic of the split-mode exchange;
    torch.distributed all_gather supplies `stats_list` across ranks).  Pure tensor glue on any device."""
    st = torch.stack(list(stats_list), dim=0)              # [R, B, NP, M+2]
    m = st[..., 0]
    m_all = m.max(dim=0).values
    scale = torch.exp(m - m_all.unsqueeze(0))              # [R, B, NP]
    Z = (st[..., 1] * scale).sum(0)
    A = (st[..., 2:] * scale.unsqueeze(-1)).sum(0)
    return torch.cat([m_all.unsqueeze(-1), Z.unsqueeze(-1), A], dim=-1)


def fk_link_positions(fk, q):
    """Link-frame origins [N, L, 3] of configurations q [N, n] for a robots.SerialChainFK (CUDA FK code)."""
    lib = _lib.load()
    _req(q, "q")
    n = fk.n_dofs
    if q.dim() != 2 or q.shape[1] != n:
        raise ValueError("q must be [N, %d]" % n)
    d = _lib.CostDesc()
    d.n_frames = len(fk.joint)
    d.include_base = 1 if fk.include_base else 0
    for f in range(len(fk.joint)):
        for k in range(9):
            d.chain_R[f][k] = fk.R[f][k]
        for k in range(3):
            d.chain_p[f][k] = fk.xyz[f][k]
        d.chain_joint[f] = fk.joint[f]
    pos = torch.empty(q.shape[0], fk.num_links, 3, dtype=q.dtype, device=q.device)
    with torch.cuda.device(q.device):
        _lib.check(lib.sgpmp_fk_link_positions(C.byref(d), n, _DT[q.dtype], q.shape[0], _ptr(q), _ptr(pos), _stream()),
                   "sgpmp_fk_link_positions")
    return pos


def select_plans(shape, desc, means, costs, n_interp, margin, want_dense=True):
    """Collision check of every particle mean at P = (T-1)(n_interp+1)+1 states (support states and the GP prior's interpolation
    between them) and the cheapest collision-free mean of each problem.  means [B,NP,T,d], costs [B,NP] (the ranking cost).
    Returns dict(clearance [B,NP], hits [B,NP] int32, particle [B] int32, ok [B] int32, plan [B,T,d], dense [B,P,d] or None)."""
    lib = _lib.load()
    B, NP, T, d = shape.B, shape.G * shape.K, shape.T, 2 * shape.n_dof
    dt, dev = means.dtype, means.device
    _req(means, "means", None, (B, NP, T, d))
    _req(costs, "costs", dt, (B, NP))
    P = (T - 1) * (max(int(n_interp), 0) + 1) + 1          # an n_interp out of range is rejected by the library
    i32 = dict(dtype=torch.int32, device=dev)
    out = dict(clearance=torch.empty(B, NP, dtype=dt, device=dev), hits=torch.empty(B, NP, **i32), particle=torch.empty(B, **i32),
               ok=torch.empty(B, **i32), plan=torch.empty(B, T, d, dtype=dt, device=dev),
               dense=torch.empty(B, P, d, dtype=dt, device=dev) if want_dense else None)
    with _on_device(dev):
        _lib.check(lib.sgpmp_select_plans(C.byref(shape), C.byref(desc), int(n_interp), float(margin), _ptr(means), _ptr(costs),
                                          _ptr(out["clearance"]), _ptr(out["hits"]), _ptr(out["particle"]), _ptr(out["ok"]),
                                          _ptr(out["plan"]), _ptr(out["dense"]), _stream()), "sgpmp_select_plans")
    return out


_GPMP_METHODS = {'inverse': _lib.GPMP_INVERSE, 'cholesky': _lib.GPMP_CHOLESKY}


def gpmp_step(shape, desc, D, O, means, delta, trust_region, method, step_size, n_iters=1, want_d_theta=True):
    """n_iters Gauss-Newton GPMP iterations (planner.py:575-600) on `means` [B,NP,T,d], in place.
    D [T,3], O [T-1,4]: float64 blocks of the start/GP/goal normal equations (planner.prior_blocks with the COST sigmas).
    Returns (costs [B,NP] = b^T K b of the last linear system, d_theta [B,NP,T,d] of the last iteration or None)."""
    lib = _lib.load()
    B, NP, T, d = shape.B, shape.G * shape.K, shape.T, 2 * shape.n_dof
    _req(means, "means", None, (B, NP, T, d))
    _req(D, "D", torch.float64, (T, 3))
    _req(O, "O", torch.float64, (T - 1, 4))
    if method not in _GPMP_METHODS:
        raise NotImplementedError("solver method %r (the reference knows 'inverse' and 'cholesky', planner.py:619-633)" % (method,))
    m = _GPMP_METHODS[method]
    dev = means.device
    nbytes = int(lib.sgpmp_gpmp_workspace_bytes(C.byref(shape), m))
    ws = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=dev)
    not_pd = torch.zeros(B * NP, dtype=torch.int32, device=dev)
    costs = torch.empty(B, NP, dtype=means.dtype, device=dev)
    d_theta = torch.empty_like(means) if want_d_theta else None
    with torch.cuda.device(dev):
        _lib.check(lib.sgpmp_gpmp_step(C.byref(shape), C.byref(desc), _ptr(D), _ptr(O), float(delta), 1 if trust_region else 0, m,
                                       float(step_size), int(n_iters), _ptr(means), _ptr(d_theta), _ptr(costs), _ptr(ws),
                                       nbytes, _ptr(not_pd), _stream()), "sgpmp_gpmp_step")
    return costs, d_theta, not_pd


def weighted_cov(shape, samples, means, weights, tensor_cores=True):
    """cov[b,p] = sum_s w_s (x_s - mu)(x_s - mu)^T  ->  [B,NP,M,M].  fp32 runs on the tensor cores (tcgen05, 3xTF32) unless
    tensor_cores=False; fp64 always on the CUDA cores.  No reference counterpart (diagnostic)."""
    lib = _lib.load()
    B, NP, T, d, S = shape.B, shape.G * shape.K, shape.T, 2 * shape.n_dof, shape.S
    dt = samples.dtype
    _req(samples, "samples", None, (B, NP, T, d, S))
    _req(means, "means", dt, (B, NP, T, d))
    _req(weights, "weights", dt, (B, NP, S))
    M = T * d
    if B * NP * M * M * samples.element_size() > 32 * 2 ** 30:
        raise ValueError("weighted_cov: the [B,NP,M,M] output would take %.1f GiB" % (B * NP * M * M * samples.element_size() / 2 ** 30))
    cov = torch.empty(B, NP, M, M, dtype=dt, device=samples.device)
    with torch.cuda.device(samples.device):
        _lib.check(lib.sgpmp_weighted_cov(C.byref(shape), _ptr(samples), _ptr(means), _ptr(weights), _ptr(cov),
                                          1 if tensor_cores else 0, _stream()), "sgpmp_weighted_cov")
    return cov


def sample_dense_tc(shape, tables, means, eps_in):
    """K2 as the reference formulates it — x = mu + L eps with the dense per-DoF scale_tril — on the tcgen05 tensor cores
    (3xTF32).  A measured comparison point for the banded recurrence of `sample()`, not the product path.  fp32, eps required."""
    lib = _lib.load()
    B, NP, T, d, S = shape.B, shape.G * shape.K, shape.T, 2 * shape.n_dof, shape.S
    _req(means, "means", torch.float32, (B, NP, T, d))
    _req(eps_in, "eps_in", torch.float32, (B, NP, T, d, S))
    L1 = prior_dense_L(tables, 1, torch.float32)                      # [2T, 2T]
    out = torch.empty_like(eps_in)
    with torch.cuda.device(means.device):
        _lib.check(lib.sgpmp_sample_dense_tc(C.byref(shape), _ptr(L1), _ptr(means), _ptr(eps_in), _ptr(out), _stream()), "sgpmp_sample_dense_tc")
    return out
