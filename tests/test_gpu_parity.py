"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI, against
 (1) the committed golden vectors produced by the unmodified reference,
 (2) the plain-C oracle on seeded inputs,
 (3) the compiled reference itself when oracle/_ref/libcpi_ref.so travelled with the snapshot,
 (4) size-independent properties at BASELINE.json's full sizes."""
import numpy as np
import pytest

from cpi_b200 import synth
from parity import compare_records, window_band

pytestmark = pytest.mark.gpu
CASES = ("cam200", "real200", "real100", "real400", "synth200", "edge")
MODES = [(1, 0), (1, 1), (2, 0), (2, 1), (2, 2), (2, 3)]
# fp32-storage variant (dtype 32): no fp32 reference exists; gates = 2x the worst error observed on B200 against the fp64 oracle on the
# same float-rounded inputs (DESIGN.md section 3a).  R/alpha/beta/J/H: fp64 arithmetic, float output rounding; P: fp32 RK4.
FP32_GATES = {1: dict(R=1.5e-7, alpha=1.5e-7, beta=1.5e-7, J_q=1.5e-7, J_a=1.5e-7, J_b=1.5e-7, H_a=1.5e-7, H_b=1.5e-7, P=6e-7, P_block=6e-7),
              2: dict(R=1.5e-7, alpha=1.5e-7, beta=1.5e-7, J_q=1.5e-7, J_a=1.5e-7, J_b=1.5e-7, H_a=1.5e-7, H_b=1.5e-7, O_a=1.5e-7, O_b=1.5e-7, P=1e-6, P_block=1e-6)}
# observed on B200 (profiles/r02_parity_vs_reference.json), model 1: R 6.4e-8, alpha/beta 5.1e-8, J/H 5.5e-8, P 2.3e-7, worst 3x3 block of P 2.9e-7:
# with the state accumulated in fp64 even the fp32 variant meets the north_star's 1e-6 on P, block-wise.


def _inputs(G, name, flags):
    avg = bool(flags & 1)
    S = G[f"{name}/samples_avg"] if avg else G[f"{name}/samples"]
    off = G[f"{name}/offsets_avg"] if avg else G[f"{name}/offsets"]
    return S, off, G[f"{name}/lin"]


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("model,flags", MODES)
def test_cuda_matches_golden(cuda, golden, name, model, flags):
    from cpi_b200 import preint
    G = golden["preint"]
    S, off, lin = _inputs(G, name, flags)
    ref = G[f"{name}/records_m{model}_f{flags}"]
    got = preint.preintegrate_host(model, S, lin, G["sigmas"], flags, offsets=off)
    steps = np.diff(off) - (1 if flags & 1 else 0)
    worst = compare_records(got, ref, model, in_band=window_band(S, off, lin), has_steps=steps > 0)
    print(name, model, flags, {k: f"{v:.1e}" for k, v in worst.items()})


@pytest.mark.parametrize("model,flags", MODES)
def test_cuda_matches_oracle_seeded(cuda, oracle, model, flags):
    """Device-pointer entry point on the bench distribution (incl. forced small_w / zero-w / dt=0 windows)."""
    from cpi_b200 import preint
    torch = cuda
    n, ns = 2100, 60                       # > 148 windows per SM-wave boundary effects: ragged last block
    S, L = synth.make_windows(n, ns, rate=200.0, first_window=0, imu_avg=bool(flags & 1))
    got = preint.preintegrate(model, torch.from_numpy(S).cuda(), torch.from_numpy(L).cuda(), synth.SIGMAS, flags, ns=ns)
    torch.cuda.synchronize()
    got = got.cpu().numpy()
    sel = np.r_[0:64, 1000:1040, n - 40:n]
    ref = oracle.preintegrate(model, S[sel], L[sel], synth.SIGMAS, flags, ns=ns, nthreads=8)
    ent = S.shape[1]
    off = np.arange(len(sel) + 1, dtype=np.int64) * ent
    compare_records(got[sel], ref, model, in_band=window_band(S[sel].reshape(-1, 7), off, L[sel]))


@pytest.mark.parametrize("model", [1, 2])
def test_cuda_matches_reference_live(cuda, oracle, model):
    """Against the compiled reference (oracle/_ref), or the C oracle where the reference was not built: the oracle is pinned to the
    reference's golden records by test_oracle.py."""
    from cpi_b200 import preint
    from oracle import oracle as om
    reference = om.Reference() if om.Reference.available() else oracle
    S, L = synth.make_windows(500, 200 if model == 1 else 400, rate=200.0 if model == 1 else 400.0, first_window=123456)
    ns = S.shape[1]
    got = preint.preintegrate_host(model, S, L, synth.SIGMAS, 0, ns=ns)
    ref = reference.preintegrate(model, S, L, synth.SIGMAS, 0, ns=ns, nthreads=16)
    off = np.arange(501, dtype=np.int64) * ns
    worst = compare_records(got, ref, model, in_band=window_band(S.reshape(-1, 7), off, L))
    print(model, {k: f"{v:.1e}" for k, v in worst.items()})


def test_ragged_and_empty_batches(cuda, oracle):
    from cpi_b200 import preint
    rng = np.random.default_rng(11)
    S, L = synth.make_windows(300, 50)
    lens = rng.integers(0, 51, size=300); lens[:5] = [0, 1, 50, 0, 2]
    wins = [S[i, :lens[i]] for i in range(300)]
    off = np.zeros(301, dtype=np.int64); off[1:] = np.cumsum(lens)
    Sx = np.concatenate(wins)
    for model in (1, 2):
        got = preint.preintegrate_host(model, Sx, L, synth.SIGMAS, 0, offsets=off)
        ref = oracle.preintegrate(model, Sx, L, synth.SIGMAS, 0, offsets=off, nthreads=8)
        compare_records(got, ref, model, in_band=window_band(Sx, off, L), has_steps=lens > 0)
        assert np.array_equal(got[0, 4:13], np.eye(3).reshape(-1)) and np.all(got[0, 13:] == 0) and np.array_equal(got[0, 0:4], [0, 0, 0, 1])
    assert preint.preintegrate_host(1, np.zeros((0, 7)), np.zeros((0, 13)), synth.SIGMAS, 0, ns=10).shape == (0, 290)


@pytest.mark.parametrize("model", [1, 2])
def test_factor_eval_matches_golden(cuda, golden, model):
    from cpi_b200 import factor
    F = golden["factor"]
    X, rec, lin = F[f"m{model}/states"], F[f"m{model}/records"], F[f"m{model}/lin"]
    for idx, suffix in ((None, ""), ((F[f"m{model}/idx_i"], F[f"m{model}/idx_j"]), "_idx")):
        e, H1, H2 = factor.factor_eval_host(model, X, rec, lin, *(idx or (None, None)))
        for got, key in ((e, "e"), (H1, "H1"), (H2, "H2")):
            ref = F[f"m{model}/{key}{suffix}"]
            err = np.max(np.abs(got - ref))
            assert err <= 1e-12 * max(1.0, np.max(np.abs(ref))), (key, err)
            assert np.array_equal(got == 0, ref == 0) or key == "e"      # structural zeros of H1/H2 are exact zeros
    e_only, h1, h2 = factor.factor_eval_host(model, X, rec, lin, want_H1=False, want_H2=False)
    assert h1 is None and h2 is None and np.max(np.abs(e_only - F[f"m{model}/e"])) <= 1e-12 * 10
    got = factor.retract(X, F[f"m{model}/xi"])
    assert np.max(np.abs(got - F[f"m{model}/retracted"])) <= 1e-14
    # predict: against the oracle restatement of getpredictedstate (GraphSolver_IMU.cpp:263-307)


@pytest.mark.parametrize("model", [1, 2])
def test_factor_chain_5k_and_predict(cuda, oracle, model):
    """Config 5 shape: 5k-keyframe chain, every factor evaluated on device; parity vs the oracle on all of them."""
    from cpi_b200 import preint, factor
    n = 4999
    S, L = synth.make_windows(n, 20, rate=200.0, first_window=9000)
    rec = preint.preintegrate_host(model, S, L, synth.SIGMAS, 0, ns=20)
    X = synth.make_states(rec, L, model)
    e, H1, H2 = factor.factor_eval_host(model, X, rec, L)
    eo, H1o, H2o = oracle.factor_eval(model, X, rec, L, nthreads=8)
    for got, ref in ((e, eo), (H1, H1o), (H2, H2o)):
        assert np.max(np.abs(got - ref)) <= 1e-11 * max(1.0, np.max(np.abs(ref)))
    pred = factor.predict_state(model, X[:-1], rec, L)
    assert np.max(np.abs(pred - oracle.predict_state(model, X[:-1], rec, L))) <= 1e-11 * np.max(np.abs(X))


def test_reference_shaped_objects(cuda, golden):
    """The CpiBase-shaped facade: feed_IMU per sample, finalize, read the public fields -- vs the reference's records."""
    from cpi_b200.preint import CpiV1, CpiV2, flush
    from cpi_b200.factor import ImuFactorCPIv1, ImuFactorCPIv2, JPLNavState
    G = golden["preint"]
    S, off, lin = G["cam200/samples"], G["cam200/offsets"], G["cam200/lin"]
    sg = G["sigmas"]
    objs = []
    for model, cls in ((1, CpiV1), (2, CpiV2)):
        for i in range(6):
            c = cls(*sg)
            c.setLinearizationPoints(lin[i, 0:3], lin[i, 3:6], lin[i, 6:10], lin[i, 10:13])
            c.imu_avg = False
            t = 0.0
            for s in S[off[i]:off[i + 1]]:
                c.feed_IMU(t, t + s[6], s[0:3], s[3:6], s[0:3], s[3:6])
                t += s[6]
            objs.append((model, i, c))
    flush([c for _, _, c in objs])
    for model, i, c in objs:
        ref = G[f"cam200/records_m{model}_f0"][i]
        # feed_IMU differences t_1 - t_0 on the host, so dt differs from the fixture's by an ulp: north_star gates
        compare_records(c.record()[None], ref[None], model, tol_mean=1e-9)
        assert c.P_meas.shape == (15, 15) and np.array_equal(c.P_meas, c.P_meas.T)
        assert abs(c.DT - ref[19]) < 1e-12
    # the factor facade: ctor argument order of the reference, evaluateError with optional Jacobians
    F = golden["factor"]
    for model in (1, 2):
        X, rec, l = F[f"m{model}/states"], F[f"m{model}/records"], F[f"m{model}/lin"]
        r = rec[3]
        m = lambda a, b, sh: r[a:b].reshape(sh, order="F")
        args = [m(65, 290, (15, 15)), r[19], l[3, 10:13], r[13:16], r[16:19], r[0:4]]
        if model == 2:
            args.append(l[3, 6:10])
        args += [l[3, 3:6], l[3, 0:3], m(20, 29, (3, 3)), m(38, 47, (3, 3)), m(29, 38, (3, 3)), m(56, 65, (3, 3)), m(47, 56, (3, 3))]
        if model == 2:
            args += [m(299, 308, (3, 3)), m(290, 299, (3, 3))]
        fac = (ImuFactorCPIv1 if model == 1 else ImuFactorCPIv2)(3, 4, *args)
        xi, xj = JPLNavState.from_vector(X[3]), JPLNavState.from_vector(X[4])
        e, H1, H2 = fac.evaluateError(xi, xj, True, True)
        assert np.max(np.abs(e - F[f"m{model}/e"][3])) <= 1e-12 * 10
        assert np.max(np.abs(H1.reshape(-1, order="F") - F[f"m{model}/H1"][3])) <= 1e-12 * 10
        assert np.max(np.abs(H2.reshape(-1, order="F") - F[f"m{model}/H2"][3])) <= 1e-12
        assert np.array_equal(fac.evaluateError(xi, xj), e)


def test_full_size_properties(cuda, oracle):
    """BASELINE configs[1]: 10k windows x 200 samples, model 1, fp64 -- properties that do not need a 10k-window oracle run."""
    from cpi_b200 import preint
    torch = cuda
    n, ns = 10000, 200
    S, L = synth.make_windows(n, ns, rate=200.0)
    dS, dL = torch.from_numpy(S).cuda(), torch.from_numpy(L).cuda()
    rec = preint.preintegrate(1, dS, dL, synth.SIGMAS, 0, ns=ns)
    # (a) shard invariance: any contiguous split gives bit-identical records (windows are independent)
    parts = [preint.preintegrate(1, dS[a:b].contiguous(), dL[a:b].contiguous(), synth.SIGMAS, 0, ns=ns) for a, b in ((0, 3333), (3333, 7000), (7000, n))]
    torch.cuda.synchronize()
    assert torch.equal(rec, torch.cat(parts))
    r = rec.cpu().numpy()
    assert np.all(np.isfinite(r))
    # (b) DT is the plain running sum of dt; R orthonormal; q consistent with R; P symmetric with the two structural zero blocks
    dts = np.zeros(n)
    for i in range(ns):
        dts += S[:, i, 6]
    assert np.array_equal(r[:, 19], dts)
    R = r[:, 4:13].reshape(n, 3, 3).transpose(0, 2, 1)
    assert np.max(np.abs(R @ R.transpose(0, 2, 1) - np.eye(3))) < 1e-12
    P = r[:, 65:290].reshape(n, 15, 15).transpose(0, 2, 1)
    assert np.array_equal(P, P.transpose(0, 2, 1))
    assert np.all(P[:, 0:6, 9:12] == 0) and np.all(np.linalg.eigvalsh(P[::97]) > -1e-18)
    # (c) bg/ba diagonal blocks are sigma^2 * DT * I up to rounding of the running sum
    assert np.allclose(P[:, 3, 3], synth.SIGMAS[1] ** 2 * dts, rtol=1e-12) and np.allclose(P[:, 9, 9], synth.SIGMAS[3] ** 2 * dts, rtol=1e-12)
    # (d) spot parity on a stride through the batch (includes the forced small_w / zero / dt=0 windows)
    mag = np.linalg.norm(S[:, :, 0:3] - L[:, None, 0:3], axis=2)
    special = np.where((mag.max(axis=1) < 0.0088) | (S[:, :, 6].min(axis=1) == 0))[0][:24]
    sel = np.unique(np.r_[np.arange(0, n, 211), special])
    ref = oracle.preintegrate(1, S[sel], L[sel], synth.SIGMAS, 0, ns=ns, nthreads=16)
    off = np.arange(len(sel) + 1, dtype=np.int64) * ns
    worst = compare_records(r[sel], ref, 1, in_band=window_band(S[sel].reshape(-1, 7), off, L[sel]))
    print({k: f"{v:.1e}" for k, v in worst.items()})


def test_cpp_facade_against_reference_headers(cuda):
    """include/cpi_b200/CpiGpu.h (CpiV1Gpu / CpiV2Gpu : CpiBase) vs the reference's own CpiV1 / CpiV2 compiled into the same
    binary (tests/cpp/test_facade, prebuilt where /root/reference exists)."""
    import os, subprocess
    exe = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cpp", "test_facade")
    if not os.path.exists(exe):
        pytest.skip("tests/cpp/test_facade not built (needs the reference headers at build time)")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    print(r.stdout, r.stderr)
    assert r.returncode == 0 and "FACADE OK" in r.stdout


def test_cpp_factor_facade_against_reference_factors(cuda):
    """include/cpi_b200/ImuFactorGpu.h (ImuFactorCPIv1Gpu / ImuFactorCPIv2Gpu : NoiseModelFactor2<JPLNavState, JPLNavState>) vs the
    reference's own ImuFactorCPIv1.cpp / ImuFactorCPIv2.cpp compiled unmodified into the same binary (against oracle/gtsam_stub):
    e, H1, H2 per factor through the per-factor path and through the graph-level batch (tests/cpp/test_factor_facade)."""
    import os, subprocess
    exe = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cpp", "test_factor_facade")
    if not os.path.exists(exe):
        pytest.skip("tests/cpp/test_factor_facade not built (needs the reference sources at build time)")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    print(r.stdout, r.stderr)
    assert r.returncode == 0 and "FACTOR FACADE OK" in r.stdout


@pytest.mark.parametrize("model,flags", [(1, 0), (2, 0), (2, 2), (1, 1)])
def test_fp32_storage_variant(cuda, oracle, model, flags):
    """dtype 32 (BASELINE configs[3]): float samples / lin / records, covariance tile and its RK4 in fp32, rotation chain, closed-form
    coefficients, means and Jacobians in fp64 (the closed forms cannot be evaluated in fp32, SURVEY section 7).  No fp32 reference
    exists (the reference is double-only): the gate is the fp64 oracle ON THE SAME float-rounded inputs, with fp32-level tolerances
    established empirically and reported in DESIGN.md."""
    from cpi_b200 import preint
    n, ns = 600, 200
    S, L = synth.make_windows(n, ns, rate=200.0, first_window=4242, imu_avg=bool(flags & 1))
    S32, L32 = S.astype(np.float32), L.astype(np.float32)
    got = preint.preintegrate_host(model, S32, L32, synth.SIGMAS, flags, ns=ns)
    assert got.dtype == np.float32 and np.all(np.isfinite(got))
    ref = oracle.preintegrate(model, S32.astype(np.float64), L32.astype(np.float64), synth.SIGMAS, flags, ns=ns, nthreads=16)
    g64 = got.astype(np.float64)
    from parity import fp32_errors
    worst = fp32_errors(got, ref)
    print(model, flags, {k: f"{v:.1e}" for k, v in worst.items()})
    # the imu_avg / analytic modes run on the round-1 lane-per-window kernels (float tile, float state): their P gate is the round-1 one
    legacy = bool(flags)
    for k, gate in FP32_GATES[model].items():
        g = gate if not (legacy and k in ("P", "P_block")) else 2e-4
        g = g if not (legacy and model == 2 and k in ("J_q", "J_a", "J_b", "H_a", "H_b", "O_a", "O_b")) else 5e-6
        assert worst[k] <= g, (k, worst[k], g)
    P = g64[:, 65:290].reshape(n, 15, 15)
    assert np.array_equal(P, P.transpose(0, 2, 1)) and np.all(P[:, 0:6, 9:12] == 0)
    # device-pointer entry point, float tensors
    torch = cuda
    d = preint.preintegrate(model, torch.from_numpy(S32).cuda(), torch.from_numpy(L32).cuda(), synth.SIGMAS, flags, ns=ns)
    torch.cuda.synchronize()
    assert d.dtype == torch.float32 and np.array_equal(d.cpu().numpy(), got)


@pytest.mark.parametrize("model,dtype", [(1, np.float64), (2, np.float64), (1, np.float32)])
def test_chunk_pipelined_host_path_is_bitwise_the_single_launch(cuda, model, dtype):
    """cpi_preintegrate_batch_host pipelines big batches in whole-window chunks (H2D / kernel / D2H overlap, chunk kernels co-resident
    on the SMs): the same bits as one launch.  Ragged windows with odd lengths exercise the 8-byte (4-byte for fp32) misaligned TMA window starts."""
    from cpi_b200 import preint
    torch = cuda
    rng = np.random.default_rng(5)
    n = 3000
    S, L = synth.make_windows(n, 200, first_window=777)
    lens = rng.integers(150, 201, size=n)
    off = np.zeros(n + 1, dtype=np.int64); off[1:] = np.cumsum(lens)
    Sx = np.concatenate([S[i, :lens[i]] for i in range(n)]).astype(dtype)
    Lx = L.astype(dtype)
    assert Sx.nbytes >= 24 << 20 or dtype == np.float32
    host = preint.preintegrate_host(model, Sx, Lx, synth.SIGMAS, 0, offsets=off)
    dev = preint.preintegrate(model, torch.from_numpy(Sx).cuda(), torch.from_numpy(Lx).cuda(), synth.SIGMAS, 0, offsets=torch.from_numpy(off).cuda())
    torch.cuda.synchronize()
    assert np.array_equal(host, dev.cpu().numpy())
    # uniform layout through the same path
    Su = S.astype(dtype)
    host_u = preint.preintegrate_host(model, Su, Lx, synth.SIGMAS, 0, ns=200)
    dev_u = preint.preintegrate(model, torch.from_numpy(Su).cuda(), torch.from_numpy(Lx).cuda(), synth.SIGMAS, 0, ns=200)
    torch.cuda.synchronize()
    if dtype == np.float32:
        assert np.array_equal(host_u, dev_u.cpu().numpy())
    else:       # fp64 + uniform layout: the tail of the batch travels in sample segments through continuation kernels (rounding-level differences)
        _close_records(host_u, dev_u.cpu().numpy(), 1e-12)


@pytest.mark.parametrize("model", [1, 2])
def test_factor_hessian_against_dense_cpu_solve(cuda, model):
    """Information-form linearisation (SURVEY 8f rank 1).  GTSAM is not in the reference tree: PARITY UNPINNED, validated against a
    dense numpy solve (Jacobi-scaled: cond(P_meas) ~ 1e7 but cond(D P D) ~ 25).  Observed on B200: 2e-15; gate 1e-10 per block."""
    from cpi_b200 import preint, factor
    n = 300
    S, L = synth.make_windows(n, 60, rate=200.0, first_window=31337, special=False)
    rec = preint.preintegrate_host(model, S, L, synth.SIGMAS, 0, ns=60)
    X = synth.make_states(rec, L, model)
    e, H1, H2 = factor.factor_eval_host(model, X, rec, L)
    G11, G12, G22, g1, g2, f = factor.factor_hessian(model, rec, e, H1, H2)
    worst = 0.0
    for i in range(n):
        P = rec[i, 65:290].reshape(15, 15, order="F")
        h1 = H1[i].reshape(15, 15, order="F"); h2 = H2[i].reshape(15, 15, order="F")
        # scaled solve for a fair CPU answer: D P D with D = diag(P)^-1/2 is well conditioned
        d = 1.0 / np.sqrt(np.diag(P)); Ps = P * d[:, None] * d[None, :]
        W = (np.linalg.inv(Ps) * d[:, None]) * d[None, :]
        ref = dict(G11=h1.T @ W @ h1, G12=h1.T @ W @ h2, G22=h2.T @ W @ h2, g1=-h1.T @ W @ e[i], g2=-h2.T @ W @ e[i], f=e[i] @ W @ e[i])
        got = dict(G11=G11[i].reshape(15, 15, order="F"), G12=G12[i].reshape(15, 15, order="F"), G22=G22[i].reshape(15, 15, order="F"), g1=g1[i], g2=g2[i], f=f[i])
        for k in ref:
            err = np.linalg.norm(got[k] - ref[k]) / max(np.linalg.norm(ref[k]), 1e-300)
            worst = max(worst, err)
            assert err <= 1e-10, (i, k, err)
        assert np.allclose(got["G11"], got["G11"].T, rtol=1e-12, atol=0) and np.allclose(got["G22"], got["G22"].T, rtol=1e-12, atol=0)
    print("worst relative block error", worst)
    # a zero-step window has P = 0: NaN outputs, no crash
    rec0 = rec[:4].copy(); rec0[1, 65:290] = 0.0
    out = factor.factor_hessian(model, rec0, e[:4], H1[:4], H2[:4])
    assert np.isnan(out[5][1]) and np.all(np.isfinite(out[5][[0, 2, 3]]))


def test_sharded_entry_point_on_device(cuda):
    """cpi_b200.shard.preintegrate_sharded with the real kernel (single process = world size 1; the N > 1 partition / padding /
    all-gather logic is covered by the gloo tests in test_shard.py and by bench.py --gpus N)."""
    from cpi_b200 import preint, shard
    S, L = synth.make_windows(500, 40, first_window=2024)
    got = shard.preintegrate_sharded(2, S.reshape(-1, 7), L, synth.SIGMAS, 0, ns=40)
    cuda.cuda.synchronize()
    assert np.array_equal(got.cpu().numpy(), preint.preintegrate_host(2, S, L, synth.SIGMAS, 0, ns=40))


def _sample_of_windows(n, cap, S, L):
    """First CTA, a CTA in the middle, the last full CTA, the last partial CTA, a stride through the batch, every forced special
    window (small_w / zero w_hat / dt = 0)."""
    mag = np.linalg.norm(S[:, :, 0:3].astype(np.float64) - L[:, None, 0:3].astype(np.float64), axis=2)
    special = np.where((mag.max(axis=1) < 0.0088) | (S[:, :, 6].min(axis=1) == 0))[0][:40]
    last_full = (n // cap - 1) * cap
    mid = (n // cap // 2) * cap
    return np.unique(np.r_[0:cap, mid:mid + cap, last_full:last_full + cap, (n // cap) * cap:n, np.arange(0, n, 401), special]).astype(np.int64)


def _close_records(a, b, tol):
    """Every record field of a within tol (relative Frobenius, per window) of b."""
    from parity import REC
    for k, (lo, hi) in REC.items():
        if hi > a.shape[1]:
            continue
        num = np.linalg.norm(a[:, lo:hi] - b[:, lo:hi], axis=1); den = np.maximum(np.linalg.norm(b[:, lo:hi], axis=1), 1e-300)
        assert np.max(num / den) <= tol, (k, float(np.max(num / den)))


@pytest.mark.parametrize("model", [1, 2])
def test_continuation_matches_one_shot(cuda, oracle, model):
    """cpi_preintegrate_batch_continue: feeding a window's samples in several calls (the batched form of further feed_IMU calls on an
    existing object, CpiBase.h:86) gives the one-shot result to rounding; a continuation with no new samples leaves the record alone."""
    from cpi_b200 import preint
    torch = cuda
    n, ns = 1203, 61
    S, L = synth.make_windows(n, ns, rate=200.0, first_window=31000)
    dS, dL = torch.from_numpy(S).cuda(), torch.from_numpy(L).cuda()
    one = preint.preintegrate(model, dS, dL, synth.SIGMAS, 0, ns=ns)
    cuts = [0, 20, 21, 21, 47, ns]                                    # uniform segments of 20, 1, 0, 26 and 14 samples
    rec = None
    for a, b in zip(cuts[:-1], cuts[1:]):
        seg = dS[:, a:b, :].contiguous()
        if rec is None:
            rec = preint.preintegrate(model, seg, dL, synth.SIGMAS, 0, ns=b - a)
        else:
            before = rec.clone()
            rec = preint.preintegrate(model, seg, dL, synth.SIGMAS, 0, ns=b - a, continue_records=rec)
            if b == a:
                torch.cuda.synchronize()
                assert torch.equal(rec, before)
    torch.cuda.synchronize()
    _close_records(rec.cpu().numpy(), one.cpu().numpy(), 1e-12)
    # ragged continuation (CSR offsets; some windows receive nothing) against the oracle fed all samples at once
    rng = np.random.default_rng(5)
    first = rng.integers(0, ns + 1, size=n); first[:4] = [0, ns, 1, ns - 1]
    offA = np.zeros(n + 1, dtype=np.int64); offA[1:] = np.cumsum(first)
    offB = np.zeros(n + 1, dtype=np.int64); offB[1:] = np.cumsum(ns - first)
    SA = np.concatenate([S[i, :first[i]] for i in range(n)]); SB = np.concatenate([S[i, first[i]:] for i in range(n)])
    rec = preint.preintegrate(model, torch.from_numpy(SA).cuda(), dL, synth.SIGMAS, 0, offsets=torch.from_numpy(offA).cuda())
    rec = preint.preintegrate(model, torch.from_numpy(SB).cuda(), dL, synth.SIGMAS, 0, offsets=torch.from_numpy(offB).cuda(), continue_records=rec)
    torch.cuda.synchronize()
    got = rec.cpu().numpy()
    _close_records(got, one.cpu().numpy(), 1e-12)
    sel = np.r_[0:40, n - 40:n]
    ref = oracle.preintegrate(model, S[sel], L[sel], synth.SIGMAS, 0, ns=ns, nthreads=8)
    compare_records(got[sel], ref, model, in_band=window_band(S[sel].reshape(-1, 7), np.arange(len(sel) + 1, dtype=np.int64) * ns, L[sel]))
    # modes without a continuation kernel refuse
    from cpi_b200 import capi
    with pytest.raises(capi.CpiError):
        preint.preintegrate(model, dS, dL, synth.SIGMAS, preint.FLAG_IMU_AVG, ns=ns - 1, continue_records=one.clone())


@pytest.mark.parametrize("model", [1, 2])
def test_host_entry_wavefront_schedule(cuda, model, monkeypatch):
    """The host entry point's wavefront schedule (window groups x sample segments, strided tile copies + continuation kernels), with
    several geometries forced onto a small batch: every window within rounding of the device one-shot call."""
    from cpi_b200 import preint
    torch = cuda
    n, ns = 3001, 100
    S, L = synth.make_windows(n, ns, rate=200.0, first_window=77000)
    one = preint.preintegrate(model, torch.from_numpy(S).cuda(), torch.from_numpy(L).cuda(), synth.SIGMAS, 0, ns=ns).cpu().numpy()
    for spec in (None, "3,4", "1,7", "40,2", "5,64", "0,0"):       # 64 segments > ns / 2 and "0,0": whole-window chunks, bit-identical
        if spec is None:
            monkeypatch.delenv("CPI_B200_HOST_WAVE", raising=False)
        else:
            monkeypatch.setenv("CPI_B200_HOST_WAVE", spec)
        host = preint.preintegrate_host(model, S, L, synth.SIGMAS, 0, ns=ns)
        _close_records(host, one, 1e-12)
        assert np.array_equal(host, one) == (spec in ("5,64", "0,0")), spec


@pytest.mark.parametrize("model,dtype,n,ns", [(1, np.float64, 25003, 200), (1, np.float32, 25003, 200), (2, np.float64, 12037, 400), (2, np.float32, 12037, 400)])
def test_multiwave_capacity_path(cuda, oracle, model, dtype, n, ns):
    """Batches of several waves of full-capacity CTAs (25k x 200 model 1 = 313 CTAs of 80 windows; 12k x 400 model 2): the
    grid-sizing path BASELINE configs[2] / configs[3] run, compared window by window with the compiled reference (oracle/_ref; the C
    port where it did not travel) on the first / a middle / the last full / the last partial CTA, a stride and all special windows."""
    from cpi_b200 import preint
    from oracle import oracle as om
    from parity import fp32_errors
    torch = cuda
    ref_impl = om.Reference() if om.Reference.available() else oracle
    rate = 200.0 if ns == 200 else 400.0
    S, L = synth.make_windows(n, ns, rate=rate, first_window=50000)
    Sx, Lx = S.astype(dtype), L.astype(dtype)
    got = preint.preintegrate(model, torch.from_numpy(Sx).cuda(), torch.from_numpy(Lx).cuda(), synth.SIGMAS, 0, ns=ns)
    torch.cuda.synchronize()
    got = got.cpu().numpy()
    assert np.all(np.isfinite(got))
    cap = 80 if not (model == 2 and dtype == np.float64) else 60
    sel = _sample_of_windows(n, cap, Sx, Lx)
    ref = ref_impl.preintegrate(model, Sx[sel].astype(np.float64), Lx[sel].astype(np.float64), synth.SIGMAS, 0, ns=ns, nthreads=16)
    if dtype == np.float64:
        off = np.arange(len(sel) + 1, dtype=np.int64) * ns
        worst = compare_records(got[sel], ref, model, in_band=window_band(S[sel].reshape(-1, 7), off, L[sel]))
    else:
        worst = fp32_errors(got[sel], ref)
        for k, gate in FP32_GATES[model].items():
            assert worst[k] <= gate, (k, worst[k], gate)
    print(model, dtype.__name__, n, ns, len(sel), {k: f"{v:.1e}" for k, v in worst.items()})
    # host entry point: whole-window chunks give the same bits (fp32); the fp64 wavefront schedule feeds every window in segments through
    # continuation kernels (rounding-level differences: the symmetric blocks are re-symmetrised at every segment)
    host = preint.preintegrate_host(model, Sx, Lx, synth.SIGMAS, 0, ns=ns)
    if dtype == np.float32:
        assert np.array_equal(host, got)
    else:
        _close_records(host, got, 1e-12)


@pytest.mark.parametrize("model", [1, 2])
def test_whitened_form_against_numpy(cuda, model):
    """A = R_w [H1 H2], b = -R_w e with R_w = chol_upper(P^-1) (GTSAM's Gaussian::Covariance; PARITY UNPINNED, GTSAM is not in the tree)."""
    from cpi_b200 import preint, factor
    n = 200
    S, L = synth.make_windows(n, 60, rate=200.0, first_window=4711, special=False)
    rec = preint.preintegrate_host(model, S, L, synth.SIGMAS, 0, ns=60)
    X = synth.make_states(rec, L, model)
    e, H1, H2 = factor.factor_eval_host(model, X, rec, L)
    A1, A2, b = factor.factor_whiten(model, rec, e, H1, H2)
    G11, G12, G22, g1, g2, f = factor.factor_hessian(model, rec, e, H1, H2)
    worst = 0.0
    for i in range(n):
        a1 = A1[i].reshape(15, 15, order="F"); a2 = A2[i].reshape(15, 15, order="F")
        # (1) the whitened blocks reproduce the information form exactly up to rounding
        for got, ref in ((a1.T @ a1, G11[i].reshape(15, 15, order="F")), (a1.T @ a2, G12[i].reshape(15, 15, order="F")), (a2.T @ a2, G22[i].reshape(15, 15, order="F")),
                         (a1.T @ b[i], g1[i]), (a2.T @ b[i], g2[i]), (b[i] @ b[i], f[i])):
            worst = max(worst, np.linalg.norm(got - ref) / max(np.linalg.norm(ref), 1e-300))
        # (2) R_w = A1 H1^-1 is upper triangular with positive diagonal and R_w^T R_w P = I   (Jacobi-scaled: cond(P) ~ 1e7)
        P = rec[i, 65:290].reshape(15, 15, order="F"); d = 1.0 / np.sqrt(np.diag(P))
        Rw = np.linalg.solve(H1[i].reshape(15, 15, order="F").T, a1.T).T if np.linalg.cond(H1[i].reshape(15, 15, order="F")) < 1e8 else None
        if Rw is not None:
            assert np.max(np.abs(np.tril(Rw, -1))) <= 1e-6 * np.max(np.abs(Rw)) and np.all(np.diag(Rw) > 0)
            Is = (Rw / d[None, :]).T @ (Rw / d[None, :]) @ (P * d[:, None] * d[None, :])
            assert np.max(np.abs(Is - np.eye(15))) < 1e-6
    print("worst relative mismatch whitened vs information form", worst)
    assert worst <= 1e-9


def _chain_truth(Dh, Eh, bh):
    """(x_true, x_banded64): scipy's banded Cholesky of the Jacobi-scaled system, then iterative refinement with 80-bit residuals --
    the refined solution is the ground truth, the unrefined one shows what a sequential fp64 CPU elimination achieves on this system."""
    import scipy.linalg
    n = len(Dh) - 1
    N = 15 * (n + 1)
    Dm = Dh.reshape(n + 1, 15, 15).transpose(0, 2, 1)               # column-major storage -> [k, row, col]
    Em = Eh.reshape(n, 15, 15).transpose(0, 2, 1) if n else np.zeros((0, 15, 15))
    sc = 1.0 / np.sqrt(np.einsum("kii->ki", Dm).reshape(-1))
    ab = np.zeros((30, N))
    for k in range(n + 1):
        for c in range(15):
            col = 15 * k + c
            ab[0:15 - c, col] = Dm[k, c:, c]
            if k < n:
                ab[15 - c:30 - c, col] = Em[k, c, :]                 # block (k, k+1): the lower part holds E^T at rows 15(k+1).., column 15k+c
    for col in range(N):
        m = min(30, N - col)
        ab[:m, col] *= sc[col] * sc[col:col + m]
    cb = scipy.linalg.cholesky_banded(ab, lower=True)
    solve = lambda r: scipy.linalg.cho_solve_banded((cb, True), np.asarray(r, dtype=np.float64).reshape(-1) * sc).reshape(n + 1, 15) * sc.reshape(n + 1, 15)
    Dl, El, bl = Dm.astype(np.longdouble), Em.astype(np.longdouble), bh.astype(np.longdouble)

    def residual(x):
        r = bl - np.einsum("krc,kc->kr", Dl, x)
        if n:
            r[:-1] -= np.einsum("krc,kc->kr", El, x[1:])
            r[1:] -= np.einsum("kcr,kc->kr", El, x[:-1])
        return r
    x64 = solve(bh)
    x = x64.astype(np.longdouble)
    for _ in range(6):
        x = x + solve(residual(x).astype(np.float64)).astype(np.longdouble)
    return x.astype(np.float64), x64


@pytest.mark.parametrize("damping", ["lambda_I", "diagonal"])
@pytest.mark.parametrize("n", [1, 2, 3, 7, 64, 300, 4999])
def test_chain_assemble_and_block_cyclic_reduction_solve(cuda, n, damping):
    """IMU-only chain of n factors: device assembly of the block-tridiagonal normal equations + block-cyclic-reduction solve, against a
    CPU banded Cholesky of the same system refined with 80-bit residuals.  PARITY UNPINNED (the reference hands this to GTSAM's smoother,
    GraphSolver.cpp:202-203); odd / even / power-of-two chain lengths exercise every end case of the reduction.
    An IMU-only chain with one prior and lambda-I damping is close to numerically singular in fp64 for any elimination order (a plain
    banded fp64 Cholesky is ~1e-6 off at 300+ keyframes): there the gate is 'as accurate as the sequential CPU elimination', with
    Marquardt (diagonal) damping the system is well posed and the gate is absolute."""
    from cpi_b200 import preint, factor
    torch = cuda
    model = 1
    S, L = synth.make_windows(n, 20, rate=200.0, first_window=9000, special=False)
    rec = preint.preintegrate_host(model, S, L, synth.SIGMAS, 0, ns=20)
    X = synth.make_states(rec, L, model)
    dX, dR, dL = (torch.from_numpy(a).cuda() for a in (X, rec, L))
    e, H1, H2 = factor.factor_eval(model, dX, dR, dL)
    G11, G12, G22, g1, g2, f = factor.factor_hessian(model, dR, e, H1, H2)
    prior = (torch.eye(15, dtype=torch.float64, device="cuda") * 1e8).reshape(-1).contiguous()
    lam, diag = (1e-3, False) if damping == "lambda_I" else (1e-5, True)
    D, E, rhs = factor.chain_assemble(G11, G12, G22, g1, g2, lam, prior, None, diagonal_damping=diag)
    x = factor.chain_solve(D, E, rhs)
    torch.cuda.synchronize()
    Dh, Eh, bh, xh = D.cpu().numpy(), E.cpu().numpy(), rhs.cpu().numpy(), x.cpu().numpy()
    # assembly against numpy
    G11h, G12h, G22h, g1h, g2h = (t.cpu().numpy() for t in (G11, G12, G22, g1, g2))
    Dref = np.zeros((n + 1, 225)); Dref[:n] += G11h; Dref[1:] += G22h; Dref[0, ::16] += 1e8
    Dref[:, ::16] += lam * np.clip(Dref[:, ::16], 1e-6, 1e32) if diag else lam
    bref = np.zeros((n + 1, 15)); bref[:n] += g1h; bref[1:] += g2h
    assert np.array_equal(Eh, G12h) and np.allclose(Dh, Dref, rtol=1e-14, atol=0) and np.allclose(bh, bref, rtol=1e-14, atol=1e-300)
    assert np.all(np.isfinite(xh))
    xt, x64 = _chain_truth(Dh, Eh, bh)
    nt = np.linalg.norm(xt)
    err, err64 = np.linalg.norm(xh - xt) / nt, np.linalg.norm(x64 - xt) / nt
    print(n, damping, "device BCR rel err vs refined truth", err, "| plain fp64 banded Cholesky (CPU)", err64)
    assert err <= 50 * max(err64, 1e-13)         # a different elimination order: same error class as the sequential fp64 solve
    if diag:
        assert err <= 1e-9


def test_chain_lm_step_reduces_the_cost(cuda):
    """eval -> Hessian blocks -> assemble -> solve -> retract, all on device: a Gauss-Newton step on a perturbed 5k-keyframe chain must
    reduce sum e^T P^-1 e by orders of magnitude (the chain started from the exact prediction has zero residual)."""
    from cpi_b200 import preint, factor
    torch = cuda
    n = 4999
    S, L = synth.make_windows(n, 20, rate=200.0, first_window=9000, special=False)
    rec = preint.preintegrate_host(1, S, L, synth.SIGMAS, 0, ns=20)
    X = synth.make_states(rec, L, 1, perturb=False)
    rng = np.random.default_rng(3)
    Xp = X.copy(); Xp[1:, 7:10] += rng.normal(0, 1e-3, (n, 3)); Xp[1:, 13:16] += rng.normal(0, 1e-3, (n, 3)); Xp[1:, 4:7] += rng.normal(0, 1e-5, (n, 3))
    dX, dR, dL = (torch.from_numpy(a).cuda() for a in (Xp, rec, L))
    X1, dx, c0 = factor.chain_lm_step(1, dX, dR, dL)                 # defaults: lambda = 1e-5 (GTSAM's lambdaInitial), diagonal damping
    X2, dx2, c1 = factor.chain_lm_step(1, X1, dR, dL)
    X3, dx3, c2 = factor.chain_lm_step(1, X2, dR, dL)
    torch.cuda.synchronize()
    c0, c1, c2 = float(c0), float(c1), float(c2)
    print("cost", c0, c1, c2, "|dx|", float(dx.norm()), float(dx2.norm()), float(dx3.norm()))
    assert np.isfinite(c0) and c1 < 1e-3 * c0 and c2 <= c1 * 1.0001 and torch.all(torch.isfinite(X3))


def test_sharded_entry_point_on_two_gpus(cuda):
    """cpi_preintegrate_batch_sharded on two ranks (one per GPU), both exchange paths, several steps over alternating gather buffers:
    every rank's gather buffer equals what the ranks computed on their own (tools/shard_check.py under torchrun).  Skipped on one GPU."""
    import json, os, subprocess, sys
    if cuda.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29541",
                        os.path.join(root, "tools", "shard_check.py")], capture_output=True, text=True, timeout=300, cwd=root)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    rep = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert rep["mismatching_steps_over_all_ranks"] == 0
    print("peer-copy path active:", [c["peer_copies"] for c in rep["cases"] if c["registered"]])
