"""Marginal covariances of the IMU chain on the device (cpi_imu_chain_marginals: selected inversion by block cyclic reduction).

GTSAM is not in the reference tree, so the diagonal blocks Sigma_kk and the adjacent blocks Sigma_k,k+1 of A^-1 are checked against dense
inverses of random SPD block-tridiagonal systems, against the covariance a filter's forward propagation gives for an IMU chain anchored at
x_0 only (a known answer), and against banded CPU solves refined with 80-bit residuals on the full 5k-keyframe chain.  Errors are
correlation-scaled: |dSigma_kl[a, b]| / sqrt(Sigma_kk[a, a] Sigma_ll[b, b])."""
import ctypes

import numpy as np
import pytest

from cpi_b200 import capi, synth


def _launches_expected(n_states):
    nl, m = 0, n_states
    while m > 1:
        m, nl = (m + 1) // 2, nl + 1
    return 3 * nl + 1


def test_argument_validation_without_gpu():
    """Bad arguments are rejected before any CUDA call; an empty chain is a no-op."""
    lib = capi.load()
    buf = np.zeros(4 * 225)
    P = ctypes.c_void_p(buf.ctypes.data)
    assert lib.cpi_imu_chain_marginals(-1, P, P, P, P, P, None) == -1 and b"negative" in lib.cpi_last_error()
    assert lib.cpi_imu_chain_marginals_workspace(-1) == -1
    assert lib.cpi_imu_chain_marginals_workspace(5000) > 0
    for args in ((None, P, P, P, P), (P, P, None, P, P), (P, P, P, P, None), (P, None, P, P, P)):
        assert lib.cpi_imu_chain_marginals(4, *args, None) == -1 and b"null" in lib.cpi_last_error(), args
    assert lib.cpi_imu_chain_marginals(0, None, None, None, None, None, None) == 0


# ---- helpers ------------------------------------------------------------------------------------------------------------------------

def _blk(a):
    """column-major flat 15x15 block(s) -> [.., row, col]"""
    return np.asarray(a).reshape(*np.shape(a)[:-1], 15, 15).swapaxes(-1, -2)


def _corr_err(Sd, So, Rd, Ro):
    """Worst correlation-scaled error of the diagonal blocks Sd[k] and the (k, k+1) blocks So[k] against the reference blocks Rd, Ro."""
    sd = np.sqrt(np.einsum("kii->ki", Rd))
    worst = float(np.max(np.abs(Sd - Rd) / (sd[:, :, None] * sd[:, None, :])))
    if len(Ro):
        worst = max(worst, float(np.max(np.abs(So - Ro) / (sd[:-1, :, None] * sd[1:, None, :]))))
    return worst


def _dense(Dm, Em):
    n = len(Dm)
    A = np.zeros((15 * n, 15 * n))
    for k in range(n):
        A[15 * k:15 * k + 15, 15 * k:15 * k + 15] = Dm[k]
        if k + 1 < n:
            A[15 * k:15 * k + 15, 15 * k + 15:15 * k + 30] = Em[k]
            A[15 * k + 15:15 * k + 30, 15 * k:15 * k + 15] = Em[k].T
    return A


def _blocks_of(Sig, n):
    Rd = np.stack([Sig[15 * k:15 * k + 15, 15 * k:15 * k + 15] for k in range(n)])
    Ro = np.stack([Sig[15 * k:15 * k + 15, 15 * k + 15:15 * k + 30] for k in range(n - 1)]) if n > 1 else np.zeros((0, 15, 15))
    return Rd, Ro


def _banded(Dm, Em):
    """scipy's banded Cholesky of the Jacobi-scaled system (the _chain_truth approach of test_gpu_parity.py): returns solve(R [N, r])."""
    import scipy.linalg
    n = len(Dm)
    N = 15 * n
    sc = 1.0 / np.sqrt(np.einsum("kii->ki", Dm).reshape(-1))
    ab = np.zeros((30, N))
    for k in range(n):
        for c in range(15):
            col = 15 * k + c
            ab[0:15 - c, col] = Dm[k, c:, c]
            if k + 1 < n:
                ab[15 - c:30 - c, col] = Em[k, c, :]
    for col in range(N):
        m = min(30, N - col)
        ab[:m, col] *= sc[col] * sc[col:col + m]
    cb = scipy.linalg.cholesky_banded(ab, lower=True)
    return lambda R: scipy.linalg.cho_solve_banded((cb, True), R * sc[:, None]) * sc[:, None]


def _chain_system(cuda, n, model=1):
    """The real IMU chain of n factors at its linearisation point: D, E of the undamped normal equations with a 1e8 I prior on x_0."""
    from cpi_b200 import preint, factor
    torch = cuda
    S, L = synth.make_windows(n, 20, rate=200.0, first_window=9000, special=False)
    rec = preint.preintegrate_host(model, S, L, synth.SIGMAS, 0, ns=20)
    X = synth.make_states(rec, L, model)
    dX, dR, dL = (torch.from_numpy(a).cuda() for a in (X, rec, L))
    e, H1, H2 = factor.factor_eval(model, dX, dR, dL)
    G11, G12, G22, g1, g2, _ = factor.factor_hessian(model, dR, e, H1, H2)
    prior = (torch.eye(15, dtype=torch.float64, device="cuda") * 1e8).reshape(-1).contiguous()
    D, E, _ = factor.chain_assemble(G11, G12, G22, g1, g2, 0.0, prior, None)
    return (dX, dR, dL), rec, H1, H2, D, E


# ---- random SPD block-tridiagonal systems ------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 8, 17, 64, 301])
def test_selected_inversion_matches_dense_inverse(cuda, n):
    """Odd, even and power-of-two sizes: last nodes with and without a right neighbour at every level of the reduction."""
    from cpi_b200 import factor
    torch = cuda
    rng = np.random.default_rng(1000 + n)
    Em = rng.standard_normal((max(n - 1, 0), 15, 15)) * 0.3
    nrm = np.array([np.linalg.norm(e, 2) for e in Em])
    Dm = np.empty((n, 15, 15))
    for k in range(n):
        B = rng.standard_normal((15, 15))
        c = 1.0 + (nrm[k - 1] if k > 0 else 0.0) + (nrm[k] if k + 1 < n else 0.0)      # block diagonal dominance: SPD
        Dm[k] = B @ B.T / 15 + c * np.eye(15)
    s = (10.0 ** rng.uniform(-0.5, 0.5, 15 * n)).reshape(n, 15)                         # state components in different units
    Dm *= s[:, :, None] * s[:, None, :]
    Em *= s[:-1, :, None] * s[1:, None, :]
    A = _dense(Dm, Em)
    print("n", n, "cond", np.linalg.cond(A))
    Rd, Ro = _blocks_of(np.linalg.inv(A), n)
    D = torch.from_numpy(np.ascontiguousarray(Dm.swapaxes(1, 2).reshape(n, 225))).cuda()
    E = torch.from_numpy(np.ascontiguousarray(Em.swapaxes(1, 2).reshape(-1, 225))).cuda()
    before = capi.launch_count()
    Sd, So = factor.chain_marginals(D, E)
    assert capi.launch_count() - before == _launches_expected(n)
    Sd2, none = factor.chain_marginals(D, E, want_off=False)
    torch.cuda.synchronize()
    assert none is None and torch.equal(Sd, Sd2)
    Sd, So = _blk(Sd.cpu().numpy()), _blk(So.cpu().numpy())
    assert np.array_equal(Sd, Sd.swapaxes(1, 2))
    err = _corr_err(Sd, So, Rd, Ro)
    print("worst correlation-scaled error vs np.linalg.inv", err)
    assert err <= 1e-11


@pytest.mark.gpu
def test_non_positive_definite_gives_nan(cuda):
    """A negative pivot gives NaN outputs, as the chain solve does (GTSAM throws there)."""
    from cpi_b200 import factor
    torch = cuda
    D = torch.eye(15, dtype=torch.float64, device="cuda").reshape(1, 225).repeat(5, 1)
    D[3] *= -1.0
    E = torch.zeros((4, 225), dtype=torch.float64, device="cuda")
    Sd, So = factor.chain_marginals(D, E)
    torch.cuda.synchronize()
    assert torch.isnan(Sd).any()


# ---- the real IMU chain: known answer ----------------------------------------------------------------------------------------------

def _forward_propagation(rec, H1, H2, prior_sigma=1e-4):
    """Covariance of a chain anchored at x_0 only: Sigma_0 = prior_sigma^2 I, Sigma_k+1 = H2^-1 (H1 Sigma_k H1^T + P) H2^-T,
    Sigma_k,k+1 = Sigma_k Phi_k^T with Phi_k = -H2^-1 H1 (e = H1 dx_k + H2 dx_k+1 with covariance P_meas)."""
    n = len(rec)
    h1, h2, P = _blk(H1), _blk(H2), _blk(rec[:, 65:290])
    Sd = np.empty((n + 1, 15, 15)); So = np.empty((n, 15, 15))
    Sd[0] = prior_sigma ** 2 * np.eye(15)
    for k in range(n):
        Phi = -np.linalg.solve(h2[k], h1[k])
        Q = np.linalg.solve(h2[k], np.linalg.solve(h2[k], P[k]).T)         # H2^-1 P H2^-T (P symmetric)
        Sd[k + 1] = Phi @ Sd[k] @ Phi.T + 0.5 * (Q + Q.T)
        So[k] = Sd[k] @ Phi.T
    return Sd, So


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 7, 64, 300])
def test_chain_marginals_equal_forward_propagation(cuda, n):
    """Undamped chain with a 1e8 I prior on x_0: the device marginals equal the filter's forward propagation of the covariance, computed from
    the device's own H1, H2 and P_meas.  The undamped chain loses conditioning fast (cond ~2e9 at 7 factors, ~4e13 at 64; DESIGN.md
    section 5), so the gate is 50 x the error of a CPU fp64 banded Cholesky of the same system (unit block right-hand sides) against the same
    answer, and 1e-9 absolute where that CPU solve itself is within 1e-10.  chain_marginal_covariances returns the same bits."""
    from cpi_b200 import factor
    torch = cuda
    (dX, dR, dL), rec, H1, H2, D, E = _chain_system(cuda, n)
    Sd, So = factor.chain_marginals(D, E)
    Sd_w, So_w = factor.chain_marginal_covariances(1, dX, dR, dL, prior_sigma=1e-4)
    torch.cuda.synchronize()
    assert torch.equal(Sd, Sd_w) and torch.equal(So, So_w)
    Rd, Ro = _forward_propagation(rec, H1.cpu().numpy(), H2.cpu().numpy())
    Sd, So = _blk(Sd.cpu().numpy()), _blk(So.cpu().numpy())
    assert np.all(np.isfinite(Sd)) and np.array_equal(Sd, Sd.swapaxes(1, 2))
    err = _corr_err(Sd, So, Rd, Ro)
    Dm, Em = _blk(D.cpu().numpy()), _blk(E.cpu().numpy())
    Bd, Bo = _blocks_of(_banded(Dm, Em)(np.eye(15 * (n + 1))), n + 1)
    err64 = _corr_err(Bd, Bo, Rd, Ro)
    print(n, "worst correlation-scaled error vs forward propagation: device", err, "| CPU fp64 banded Cholesky", err64)
    assert err <= 50 * max(err64, 1e-13)
    if err64 <= 1e-10:
        assert err <= 1e-9


# ---- full size, well posed ----------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_full_chain_marginals_against_refined_banded_solve(cuda):
    """4 999 factors with a per-keyframe orientation / position prior added to every D block (standing in for the camera factors): the
    blocks of 40 sampled keyframes plus the first and the last against scipy's banded Cholesky refined with 80-bit residuals."""
    from cpi_b200 import factor
    torch = cuda
    n = 4999
    _, _, _, _, D, E = _chain_system(cuda, n)
    kf = torch.zeros(225, dtype=torch.float64, device="cuda")
    kf[0:3 * 16:16] = 1.0 / 1e-2 ** 2                                   # theta: 0.01 rad
    kf[12 * 16::16] = 1.0 / 0.1 ** 2                                    # p: 0.1 m
    D = D + kf
    Sd, So = factor.chain_marginals(D, E)
    torch.cuda.synchronize()
    Sd, So = _blk(Sd.cpu().numpy()), _blk(So.cpu().numpy())
    assert np.all(np.isfinite(Sd)) and np.all(np.isfinite(So)) and np.array_equal(Sd, Sd.swapaxes(1, 2))
    Dm, Em = _blk(D.cpu().numpy()), _blk(E.cpu().numpy())
    solve = _banded(Dm, Em)
    Dl, El = Dm.astype(np.longdouble), Em.astype(np.longdouble)
    ks = np.unique(np.r_[0, n, np.random.default_rng(7).choice(np.arange(1, n), 40, replace=False)])
    worst = 0.0
    for k in ks:
        R = np.zeros((15 * (n + 1), 15)); R[15 * k:15 * k + 15] = np.eye(15)      # columns of block k of A^-1
        X = solve(R)
        for _ in range(2):                                              # refinement with 80-bit residuals
            x = X.reshape(n + 1, 15, 15).astype(np.longdouble)
            r = -np.einsum("krc,kcj->krj", Dl, x)
            r[:-1] -= np.einsum("krc,kcj->krj", El, x[1:])
            r[1:] -= np.einsum("kcr,kcj->krj", El, x[:-1])
            r[k] += np.eye(15)
            X = X + solve(r.reshape(-1, 15).astype(np.float64))
        X = X.reshape(n + 1, 15, 15)                                    # X[j] = Sigma_jk
        sd = np.sqrt(np.diag(X[k]))
        e = float(np.max(np.abs(Sd[k] - X[k]) / np.outer(sd, sd)))
        if k < n:                                                       # Sigma_k,k+1 = Sigma_k+1,k^T, scaled with the device's Sigma_k+1,k+1
            s1 = np.sqrt(np.diag(Sd[k + 1]))
            e = max(e, float(np.max(np.abs(So[k] - X[k + 1].T) / np.outer(sd, s1))))
        worst = max(worst, e)
    print("worst correlation-scaled error over", len(ks), "keyframes vs refined banded solve", worst)
    assert worst <= 1e-9
