"""Host-side mirror of the GTSAM-side plug-ins of the hot path, on top of the C ABI:

    JPLNavState                      gtsam/JPLNavState.h:59-151   (value layout q, bg, v, ba, p; retract)
    ImuFactorCPIv1 / ImuFactorCPIv2  gtsam/ImuFactorCPIv1.h:55, gtsam/ImuFactorCPIv2.h:55   (ctor argument order kept)
        .evaluateError(state_i, state_j, H1=False, H2=False)      gtsam/ImuFactorCPIv1.cpp:37, ImuFactorCPIv2.cpp:38

and the batch entry points (``factor_eval``, ``predict_state``, ``retract``, the chain solve and its marginal covariances).  The residual and Jacobians are UNWHITENED,
exactly what evaluateError returns; GTSAM's Gaussian::Covariance(P_meas) whitening is outside the reference tree.
All arithmetic happens in libcpi_b200.so on the GPU.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import capi
from .capi import REC, REC_DOUBLES


def _ptr(a):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


def _tptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def factor_eval_host(model, states, records, lin, idx_i=None, idx_j=None, want_H1=True, want_H2=True):
    """HOST numpy in/out through ``cpi_imu_factor_eval_batch_host``.  Returns (e[n,15], H1[n,225]|None, H2[n,225]|None);
    H blocks are column-major 15x15 (reshape(15,15,order='F'))."""
    lib = capi.load()
    states = np.ascontiguousarray(states, dtype=np.float64).reshape(-1, 16)
    records = np.ascontiguousarray(records, dtype=np.float64).reshape(-1, REC_DOUBLES[model])
    lin = np.ascontiguousarray(lin, dtype=np.float64).reshape(-1, 13)
    n = records.shape[0]
    if lin.shape[0] != n:
        raise ValueError("one linearisation point per factor required")
    if (idx_i is None) != (idx_j is None):
        raise ValueError("idx_i and idx_j must both be given or both be None")
    if idx_i is not None:
        idx_i = np.ascontiguousarray(idx_i, dtype=np.int64); idx_j = np.ascontiguousarray(idx_j, dtype=np.int64)
        if idx_i.shape[0] != n or idx_j.shape[0] != n:
            raise ValueError("index arrays must have one entry per factor")
        if n and (min(idx_i.min(), idx_j.min()) < 0 or max(idx_i.max(), idx_j.max()) >= states.shape[0]):
            raise IndexError("state index out of range")
    elif states.shape[0] < n + 1:
        raise ValueError("chain indexing needs n_factors + 1 states")
    e = np.empty((n, 15)); H1 = np.empty((n, 225)) if want_H1 else None; H2 = np.empty((n, 225)) if want_H2 else None
    capi.check(lib.cpi_imu_factor_eval_batch_host(model, n, states.shape[0], _ptr(states), _ptr(idx_i), _ptr(idx_j), _ptr(records), _ptr(lin),
                                                  _ptr(e), _ptr(H1), _ptr(H2)))
    return e, H1, H2


def factor_eval(model, states, records, lin, idx_i=None, idx_j=None, want_H1=True, want_H2=True, out=None, stream=None):
    """DEVICE torch tensors (float64 / int64, contiguous).  Enqueues on ``stream`` (default: torch's current stream)."""
    import torch

    lib = capi.load()
    n = records.numel() // REC_DOUBLES[model]
    dev = records.device
    for name, t in (("states", states), ("lin", lin), ("idx_i", idx_i), ("idx_j", idx_j)):
        if t is not None and (not t.is_cuda or t.device != dev):
            raise ValueError(f"{name} must be a CUDA tensor on {dev}")
    if (idx_i is None) != (idx_j is None):
        raise ValueError("idx_i and idx_j must both be given or both be None")
    if idx_i is not None:
        if idx_i.dtype != torch.int64 or idx_j.dtype != torch.int64 or idx_i.numel() != n or idx_j.numel() != n:
            raise ValueError("idx_i / idx_j must be int64 tensors with one entry per factor")
        idx_i = idx_i.contiguous(); idx_j = idx_j.contiguous()
    if out is None:
        e = torch.empty((n, 15), dtype=torch.float64, device=dev)
        H1 = torch.empty((n, 225), dtype=torch.float64, device=dev) if want_H1 else None
        H2 = torch.empty((n, 225), dtype=torch.float64, device=dev) if want_H2 else None
    else:
        e, H1, H2 = out
    with torch.cuda.device(dev):
        st = stream if stream is not None else torch.cuda.current_stream(dev)
        capi.check(lib.cpi_imu_factor_eval_batch(model, n, _tptr(states.contiguous()), _tptr(idx_i), _tptr(idx_j), _tptr(records.contiguous()),
                                                 _tptr(lin.contiguous()), _tptr(e), _tptr(H1), _tptr(H2), ctypes.c_void_p(st.cuda_stream)))
    return e, H1, H2


def factor_hessian(model, records, e, H1, H2, stream=None):
    """Information-form linearisation (cpi_imu_factor_hessian_batch): returns (G11, G12, G22 [n,225 col-major], g1, g2 [n,15], f [n]).
    Device tensors in/out, or numpy (staged through torch).  Parity vs GTSAM unpinned (GTSAM is not in the reference tree)."""
    import torch

    lib = capi.load()
    host = isinstance(records, np.ndarray)
    if host:
        records, e, H1, H2 = (torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda() for a in (records, e, H1, H2))
    n = records.numel() // REC_DOUBLES[model]
    dev = records.device
    G11, G12, G22 = (torch.empty((n, 225), dtype=torch.float64, device=dev) for _ in range(3))
    g1, g2 = (torch.empty((n, 15), dtype=torch.float64, device=dev) for _ in range(2))
    f = torch.empty((n,), dtype=torch.float64, device=dev)
    st = stream if stream is not None else torch.cuda.current_stream()
    capi.check(lib.cpi_imu_factor_hessian_batch(model, n, _tptr(records.contiguous()), _tptr(e.contiguous()), _tptr(H1.contiguous()), _tptr(H2.contiguous()),
                                                _tptr(G11), _tptr(G12), _tptr(G22), _tptr(g1), _tptr(g2), _tptr(f), ctypes.c_void_p(st.cuda_stream)))
    out = (G11, G12, G22, g1, g2, f)
    return tuple(t.cpu().numpy() for t in out) if host else out


def factor_whiten(model, records, e, H1, H2, stream=None):
    """Explicitly whitened form (cpi_imu_factor_whiten_batch): A1 = R_w H1, A2 = R_w H2 [n,225 col-major], b = -R_w e [n,15], with
    R_w the upper Cholesky factor of P_meas^-1 (GTSAM's Gaussian::Covariance).  Device tensors in/out, or numpy.  Parity unpinned."""
    import torch

    lib = capi.load()
    host = isinstance(records, np.ndarray)
    if host:
        records, e, H1, H2 = (torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda() for a in (records, e, H1, H2))
    n = records.numel() // REC_DOUBLES[model]
    A1, A2 = (torch.empty((n, 225), dtype=torch.float64, device=records.device) for _ in range(2))
    b = torch.empty((n, 15), dtype=torch.float64, device=records.device)
    st = stream if stream is not None else torch.cuda.current_stream()
    capi.check(lib.cpi_imu_factor_whiten_batch(model, n, _tptr(records.contiguous()), _tptr(e.contiguous()), _tptr(H1.contiguous()), _tptr(H2.contiguous()),
                                               _tptr(A1), _tptr(A2), _tptr(b), ctypes.c_void_p(st.cuda_stream)))
    out = (A1, A2, b)
    return tuple(t.cpu().numpy() for t in out) if host else out


def chain_assemble(G11, G12, G22, g1, g2, lam=0.0, prior_info0=None, prior_rhs0=None, stream=None, diagonal_damping=False):
    """Block-tridiagonal normal equations of the chain x_0 .. x_n from the per-factor information blocks (cpi_imu_chain_assemble).
    Device tensors.  Damping: lam * I, or with diagonal_damping lam * clamp(diag, 1e-6, 1e32) (GTSAM's LevenbergMarquardtParams::diagonalDamping).
    Returns (D [n+1,225], E [n,225], rhs [n+1,15])."""
    import torch

    lib = capi.load()
    n = G11.shape[0]
    dev = G11.device
    D = torch.empty((n + 1, 225), dtype=torch.float64, device=dev)
    E = torch.empty((max(n, 1), 225), dtype=torch.float64, device=dev)
    rhs = torch.empty((n + 1, 15), dtype=torch.float64, device=dev)
    st = stream if stream is not None else torch.cuda.current_stream()
    capi.check(lib.cpi_imu_chain_assemble(n, _tptr(G11), _tptr(G12), _tptr(G22), _tptr(g1), _tptr(g2), float(lam), int(bool(diagonal_damping)), _tptr(prior_info0), _tptr(prior_rhs0),
                                          _tptr(D), _tptr(E), _tptr(rhs), ctypes.c_void_p(st.cuda_stream)))
    return D, E[:n], rhs


def chain_solve(D, E, rhs, stream=None, workspace=None):
    """x = A^-1 rhs for the SPD block-tridiagonal A = tridiag(E^T, D, E) by block cyclic reduction on the device (cpi_imu_chain_solve)."""
    import torch

    lib = capi.load()
    n = D.shape[0]
    x = torch.empty((n, 15), dtype=torch.float64, device=D.device)
    nbytes = int(lib.cpi_imu_chain_solve_workspace(n))
    if workspace is None or workspace.numel() * 8 < nbytes:
        workspace = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=D.device)
    st = stream if stream is not None else torch.cuda.current_stream()
    capi.check(lib.cpi_imu_chain_solve(n, _tptr(D), _tptr(E), _tptr(rhs), _tptr(x), _tptr(workspace), ctypes.c_void_p(st.cuda_stream)))
    return x


def chain_marginals(D, E, want_off=True, workspace=None, stream=None):
    """Marginal covariances of the chain (cpi_imu_chain_marginals): the diagonal blocks Sigma_kk and, with want_off, the blocks Sigma_k,k+1
    of Sigma = A^-1 for A = tridiag(E^T, D, E), by selected inversion on the device.  Device tensors D [n+1,225], E [n,225].
    Returns (S_diag [n+1,225], S_off [n,225] or None), column-major 15x15 blocks."""
    import torch

    lib = capi.load()
    n = D.shape[0]
    S_diag = torch.empty((n, 225), dtype=torch.float64, device=D.device)
    S_off = torch.empty((max(n - 1, 0), 225), dtype=torch.float64, device=D.device) if want_off else None
    nbytes = int(lib.cpi_imu_chain_marginals_workspace(n))
    if workspace is None or workspace.numel() * 8 < nbytes:
        workspace = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=D.device)
    st = stream if stream is not None else torch.cuda.current_stream()
    capi.check(lib.cpi_imu_chain_marginals(n, _tptr(D.contiguous()), _tptr(E.contiguous()), _tptr(S_diag), _tptr(S_off), _tptr(workspace),
                                           ctypes.c_void_p(st.cuda_stream)))
    return S_diag, S_off


_PRIOR = {}


def _prior_info(dev, prior_sigma):
    """1/prior_sigma^2 I (15x15, flattened) on x_0, cached per device."""
    import torch

    key = (dev, prior_sigma)
    if key not in _PRIOR:
        _PRIOR[key] = (torch.eye(15, dtype=torch.float64, device=dev) / (prior_sigma * prior_sigma)).reshape(-1).contiguous()
    return _PRIOR[key]


def chain_lm_step(model, states, records, lin, lam=1e-5, prior_sigma=1e-4, stream=None, diagonal_damping=True):
    """One damped Gauss-Newton (Levenberg-Marquardt) step of an IMU-only chain, entirely on the device:
    evaluateError for every factor -> information blocks -> block-tridiagonal assembly (prior 1/prior_sigma^2 on x_0: the
    reference initialises with cov = 1e-8 I, GraphSolver.cpp:331; Marquardt damping lam * diag by default, lam = GTSAM's lambdaInitial:
    an undamped IMU-only chain of thousands of keyframes is numerically singular in fp64) -> block-cyclic-reduction solve -> JPLNavState::retract.
    Returns (new_states, delta, cost = sum e^T P^-1 e before the step)."""
    e, H1, H2 = factor_eval(model, states, records, lin, stream=stream)
    G11, G12, G22, g1, g2, f = factor_hessian(model, records, e, H1, H2, stream=stream)
    D, E, rhs = chain_assemble(G11, G12, G22, g1, g2, lam, _prior_info(states.device, prior_sigma), None, stream=stream, diagonal_damping=diagonal_damping)
    dx = chain_solve(D, E, rhs, stream=stream)
    return retract(states, dx, stream=stream), dx, f.sum()


def chain_marginal_covariances(model, states, records, lin, prior_sigma=1e-4, stream=None):
    """Marginal covariances of an IMU-only chain at ``states``, what GTSAM's Marginals computes at an estimate: the normal equations are
    linearised there without damping (lambda = 0), with the x_0 prior of chain_lm_step, and inverted selectively on the device.
    Returns (S_diag [n+1,225]: Sigma_kk, S_off [n,225]: Sigma_k,k+1), column-major 15x15 blocks in the error-state order.
    An IMU-only chain anchored by one prior is numerically singular in fp64 beyond a few hundred keyframes (DESIGN.md section 5)."""
    e, H1, H2 = factor_eval(model, states, records, lin, stream=stream)
    G11, G12, G22, g1, g2, _ = factor_hessian(model, records, e, H1, H2, stream=stream)
    D, E, _ = chain_assemble(G11, G12, G22, g1, g2, 0.0, _prior_info(states.device, prior_sigma), None, stream=stream)
    return chain_marginals(D, E, stream=stream)


def predict_state(model, states_k, records, lin, stream=None):
    """getpredictedstate_v1/_v2 (solvers/GraphSolver_IMU.cpp:263-307), batched.  Device tensors, or numpy (staged via torch)."""
    import torch

    lib = capi.load()
    host = isinstance(states_k, np.ndarray)
    if host:
        states_k, records, lin = (torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda() for a in (states_k, records, lin))
    n = states_k.numel() // 16
    out = torch.empty((n, 16), dtype=torch.float64, device=states_k.device)
    st = stream if stream is not None else torch.cuda.current_stream()
    capi.check(lib.cpi_predict_state_batch(model, n, _tptr(states_k.contiguous()), _tptr(records.contiguous()), _tptr(lin.contiguous()), _tptr(out),
                                           ctypes.c_void_p(st.cuda_stream)))
    return out.cpu().numpy() if host else out


def retract(states, xi, stream=None):
    """JPLNavState::retract (gtsam/JPLNavState.cpp:37-71), batched."""
    import torch

    lib = capi.load()
    host = isinstance(states, np.ndarray)
    if host:
        states, xi = (torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda() for a in (states, xi))
    n = states.numel() // 16
    out = torch.empty((n, 16), dtype=torch.float64, device=states.device)
    st = stream if stream is not None else torch.cuda.current_stream()
    capi.check(lib.cpi_retract_batch(n, _tptr(states.contiguous()), _tptr(xi.contiguous()), _tptr(out), ctypes.c_void_p(st.cuda_stream)))
    return out.cpu().numpy() if host else out


class JPLNavState:
    """gtsam/JPLNavState.h:59-151: [q_GtoI(4, JPL xyzw), biasg(3), v_IinG(3), biasa(3), p_IinG(3)], dimension 15."""
    dimension = 15

    def __init__(self, q=(0, 0, 0, 1), bg=(0, 0, 0), v=(0, 0, 0), ba=(0, 0, 0), p=(0, 0, 0)):
        self._x = np.concatenate([np.asarray(a, dtype=np.float64).reshape(-1) for a in (q, bg, v, ba, p)])
        assert self._x.shape == (16,)

    @classmethod
    def from_vector(cls, x):
        x = np.asarray(x, dtype=np.float64).reshape(16)
        return cls(x[0:4], x[4:7], x[7:10], x[10:13], x[13:16])

    def vector(self): return self._x.copy()
    def q(self): return self._x[0:4].copy()
    def bg(self): return self._x[4:7].copy()
    def v(self): return self._x[7:10].copy()
    def ba(self): return self._x[10:13].copy()
    def p(self): return self._x[13:16].copy()

    def retract(self, xi):
        return JPLNavState.from_vector(retract(self._x[None], np.asarray(xi, dtype=np.float64).reshape(1, 15))[0])

    def equals(self, other, tol=1e-8):
        return bool(np.all(np.abs(self._x - other._x) <= tol))


class _ImuFactorCPI:
    model = 0

    def _pack(self, covariance, deltatime, grav, alpha, beta, q_KtoK1, q_K_lin, ba_lin, bg_lin, J_q, J_beta, J_alpha, H_beta, H_alpha,
              O_beta=None, O_alpha=None):
        rec = np.zeros(REC_DOUBLES[self.model])

        def put(name, a):
            lo, hi = REC[name]
            rec[lo:hi] = np.asarray(a, dtype=np.float64).reshape(-1, order="F")
        put("q", q_KtoK1); put("alpha", alpha); put("beta", beta); rec[19] = float(deltatime)
        put("J_q", J_q); put("J_a", J_alpha); put("J_b", J_beta); put("H_a", H_alpha); put("H_b", H_beta); put("P", covariance)
        if self.model == 2:
            put("O_a", O_alpha); put("O_b", O_beta)
        self._rec = rec
        self._lin = np.concatenate([np.asarray(bg_lin, dtype=np.float64).reshape(3), np.asarray(ba_lin, dtype=np.float64).reshape(3),
                                    np.asarray(q_K_lin, dtype=np.float64).reshape(4), np.asarray(grav, dtype=np.float64).reshape(3)])

    # accessors of the reference class (ImuFactorCPIv1.h:104-134)
    def dt(self): return float(self._rec[19])
    def m_alpha(self): return self._rec[13:16].copy()
    def m_beta(self): return self._rec[16:19].copy()
    def m_q(self): return self._rec[0:4].copy()
    def m_balin(self): return self._lin[3:6].copy()
    def m_bglin(self): return self._lin[0:3].copy()
    def gravity(self): return self._lin[10:13].copy()
    def key1(self): return self._keys[0]
    def key2(self): return self._keys[1]

    def evaluateError(self, state_i, state_j, H1=False, H2=False):
        """Returns the 15-vector error; with H1/H2 truthy returns (error, H1, H2) with 15x15 arrays (None if not asked)."""
        X = np.stack([state_i.vector(), state_j.vector()])
        e, h1, h2 = factor_eval_host(self.model, X, self._rec[None], self._lin[None], want_H1=bool(H1), want_H2=bool(H2))
        if not (H1 or H2):
            return e[0]
        return (e[0], h1[0].reshape(15, 15, order="F") if H1 else None, h2[0].reshape(15, 15, order="F") if H2 else None)

    def equals(self, other, tol=1e-9):
        return type(other) is type(self) and self._keys == other._keys and bool(
            np.all(np.abs(self._rec - other._rec) <= tol) and np.all(np.abs(self._lin - other._lin) <= tol))


class ImuFactorCPIv1(_ImuFactorCPI):
    """gtsam/ImuFactorCPIv1.h:78-82 -- argument order kept (note J_beta before J_alpha, H_beta before H_alpha)."""
    model = 1

    def __init__(self, state_i, state_j, covariance, deltatime, grav, alpha, beta, q_KtoK1, ba_lin, bg_lin, J_q, J_beta, J_alpha,
                 H_beta, H_alpha):
        self._keys = (state_i, state_j)
        self._pack(covariance, deltatime, grav, alpha, beta, q_KtoK1, np.array([0, 0, 0, 1.0]), ba_lin, bg_lin, J_q, J_beta, J_alpha,
                   H_beta, H_alpha)


class ImuFactorCPIv2(_ImuFactorCPI):
    """gtsam/ImuFactorCPIv2.h:82-86 (adds q_K_lin, O_beta, O_alpha)."""
    model = 2

    def __init__(self, state_i, state_j, covariance, deltatime, grav, alpha, beta, q_KtoK1, q_K_lin, ba_lin, bg_lin, J_q, J_beta,
                 J_alpha, H_beta, H_alpha, O_beta, O_alpha):
        self._keys = (state_i, state_j)
        self._pack(covariance, deltatime, grav, alpha, beta, q_KtoK1, q_K_lin, ba_lin, bg_lin, J_q, J_beta, J_alpha, H_beta, H_alpha,
                   O_beta, O_alpha)

    def m_qklin(self): return self._lin[6:10].copy()
