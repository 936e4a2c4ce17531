"""CPU tests: the plain-C oracle is pinned to the reference -- against the committed golden vectors (always) and against
the compiled reference itself (when oracle/_ref/libcpi_ref.so is present)."""
import numpy as np
import pytest

from cpi_b200 import synth
from parity import compare_records, window_band

CASES = ("cam200", "real200", "real100", "real400", "synth200", "edge")
TIGHT = dict(tol_mean=1e-12, tol_P=1e-12, tol_J=1e-11, tol_Ja_band=1e-9)


def _inputs(G, name, flags):
    avg = bool(flags & 1)
    S = G[f"{name}/samples_avg"] if avg else G[f"{name}/samples"]
    off = G[f"{name}/offsets_avg"] if avg else G[f"{name}/offsets"]
    return S, off, G[f"{name}/lin"]


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("model,flags", [(1, 0), (1, 1), (2, 0), (2, 1), (2, 2), (2, 3)])
def test_oracle_matches_golden(oracle, golden, name, model, flags):
    G = golden["preint"]
    S, off, lin = _inputs(G, name, flags)
    ref = G[f"{name}/records_m{model}_f{flags}"]
    got = oracle.preintegrate(model, S, lin, G["sigmas"], flags, offsets=off)
    steps = np.diff(off) - (1 if flags & 1 else 0)
    # "edge" holds a window sitting exactly ON the small_w threshold (CpiV1.h:101): a 1-ulp difference in |w_hat|
    # flips the Taylor/closed-form branch there (the two differ by ~1e-11), so that case gets the north_star gates.
    tol = {} if name == "edge" else TIGHT
    compare_records(got, ref, model, in_band=window_band(S, off, lin), has_steps=steps > 0, **tol)


@pytest.mark.parametrize("model", [1, 2])
def test_oracle_matches_reference_live(oracle, reference, model):
    S, L = synth.make_windows(48, 120, rate=200.0, first_window=5000)
    off = np.arange(49, dtype=np.int64) * 120
    got = oracle.preintegrate(model, S, L, synth.SIGMAS, 0, ns=120)
    ref = reference.preintegrate(model, S, L, synth.SIGMAS, 0, ns=120)
    compare_records(got, ref, model, in_band=window_band(S.reshape(-1, 7), off, L), **TIGHT)


@pytest.mark.parametrize("model", [1, 2])
def test_oracle_factor_matches_golden(oracle, golden, model):
    F = golden["factor"]
    X, rec, lin = F[f"m{model}/states"], F[f"m{model}/records"], F[f"m{model}/lin"]
    e, H1, H2 = oracle.factor_eval(model, X, rec, lin)
    for got, key in ((e, "e"), (H1, "H1"), (H2, "H2")):
        ref = F[f"m{model}/{key}"]
        assert np.max(np.abs(got - ref)) <= 1e-12 * max(1.0, np.max(np.abs(ref)))
    e, H1, H2 = oracle.factor_eval(model, X, rec, lin, F[f"m{model}/idx_i"], F[f"m{model}/idx_j"])
    for got, key in ((e, "e_idx"), (H1, "H1_idx"), (H2, "H2_idx")):
        ref = F[f"m{model}/{key}"]
        assert np.max(np.abs(got - ref)) <= 1e-12 * max(1.0, np.max(np.abs(ref)))
    assert np.max(np.abs(oracle.retract(X, F[f"m{model}/xi"]) - F[f"m{model}/retracted"])) <= 1e-14


def test_oracle_quat_ops_match_reference(oracle, golden):
    """Every golden record stores the reference's q = rot_2_quat(R) of its own R (CpiV1.h:358): the oracle's rot_2_quat must give the
    same quaternion on all of them.  The other helpers are compared live when oracle/_ref/libcpi_ref.so is built."""
    from oracle import oracle as om
    G = golden["preint"]
    for key in (k for k in G.files if "/records_" in k):
        for rec in G[key]:
            assert np.max(np.abs(oracle.rot_2_quat(rec[4:13]) - rec[0:4])) <= 1e-15, key
    if not om.Reference.available():
        return
    reference = om.Reference()
    rng = np.random.default_rng(3)
    for _ in range(50):
        q = rng.normal(size=4); q /= np.linalg.norm(q)
        p = rng.normal(size=4); p /= np.linalg.norm(p)
        w = rng.normal(size=3) * rng.choice([1e-9, 1e-3, 1.0, 3.0])
        R = reference.quat_2_Rot(q)
        assert np.max(np.abs(oracle.quat_2_Rot(q) - R)) <= 1e-15
        assert np.max(np.abs(oracle.rot_2_quat(R) - reference.rot_2_quat(R))) <= 1e-15
        assert np.max(np.abs(oracle.quat_multiply(q, p) - reference.quat_multiply(q, p))) <= 1e-15
        assert np.max(np.abs(oracle.Exp(w) - reference.Exp(w))) <= 8e-15  # |w| up to ~5 rad: a few ulp of O(1) entries
    assert np.array_equal(oracle.Exp(np.zeros(3)), np.eye(3).reshape(-1))


def test_known_answer_residual_at_predicted_state(oracle):
    """SURVEY 4: the residual at (x_k, predicted x_{k+1}) with biases / q at the linearisation point is ~1e-15."""
    S, L = synth.make_windows(6, 80, rate=200.0, first_window=77, special=False)
    for model in (1, 2):
        x = np.zeros((1, 16)); x[0, 0:4] = [0.1, -0.2, 0.3, 0.0]; x[0, 3] = np.sqrt(1 - 0.14); x[0, 7:10] = [1.0, -0.5, 0.2]
        for k in range(6):
            lin = L[k:k + 1].copy()
            x[0, 4:7] = lin[0, 0:3]; x[0, 10:13] = lin[0, 3:6]; lin[0, 6:10] = x[0, 0:4]
            rec = oracle.preintegrate(model, S[k], lin, synth.SIGMAS, 0, ns=80)
            x1 = oracle.predict_state(model, x, rec, lin)
            e, _, _ = oracle.factor_eval(model, np.concatenate([x, x1]), rec, lin)
            assert np.max(np.abs(e)) < 5e-13, (model, k, e)
            x = x1
