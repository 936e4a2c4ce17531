"""Timing of cpi_imu_chain_marginals (selected inversion by block cyclic reduction) on the configs[4] chain (4 999 factors) and on a
100 000-state chain (the 5k chain's factor blocks tiled), next to one LM step and the "LM step + marginal covariances" sequence.

CUDA-event times per call after warm-up (median over --reps calls; the 5k chain's working set stays in L2 between calls, the 100k chain's
~300 MB does not).  The systems carry a per-keyframe orientation / position prior on every D block, standing in for the camera factors,
so that the timed inversions are well posed.  Prints one JSON line with the device name, its power limit and the launch counts.

    python tools/chain_marginals_probe.py [--reps 200] [--warmup 20]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _time(fn, reps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in evs:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) for a, b in evs]))


def _launches(fn):
    from cpi_b200 import capi
    before = capi.launch_count()
    fn()
    return capi.launch_count() - before


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    import torch
    from cpi_b200 import capi, factor, preint, synth
    if not torch.cuda.is_available():
        raise SystemExit("chain_marginals_probe.py needs a CUDA device")
    capi.load()
    n = 4999                                                           # configs[4]: the 5k-keyframe chain of bench.py
    S, L = synth.make_windows(n, 20, rate=200.0, first_window=9000)
    rec = preint.preintegrate_host(1, S, L, synth.SIGMAS, 0, ns=20)
    X = synth.make_states(rec, L, 1)
    dX, dR, dL = (torch.from_numpy(a).cuda() for a in (X, rec, L))
    e, H1, H2 = factor.factor_eval(1, dX, dR, dL)
    G = factor.factor_hessian(1, dR, e, H1, H2)
    prior = (torch.eye(15, dtype=torch.float64, device="cuda") * 1e8).reshape(-1).contiguous()
    kf = torch.zeros(225, dtype=torch.float64, device="cuda")
    kf[0:3 * 16:16] = 1e4; kf[12 * 16::16] = 1e2                      # theta 0.01 rad, p 0.1 m on every keyframe

    out = {"tool": "chain_marginals_probe", "device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["sm_clock_max"] = [x.strip() for x in q.split(",")]
    except Exception as ex:                                            # the numbers are still device timings; say what is missing
        out["power_limit"] = f"unavailable ({ex})"
    out["timing"] = f"CUDA events, median of {args.reps} calls after {args.warmup} warm-up calls"

    for name, nf in (("chain_5k", n), ("chain_100k", 99_999)):
        Gt = [t.repeat(-(-nf // n), 1)[:nf].contiguous() for t in G[:5]]       # factor blocks tiled: a sum of PSD terms stays PSD
        D, E, _ = factor.chain_assemble(*Gt, 0.0, prior, None)
        D = (D + kf).contiguous()
        ws = torch.empty(int(capi.load().cpi_imu_chain_marginals_workspace(nf + 1)) // 8 + 1, dtype=torch.float64, device="cuda")
        call = lambda: factor.chain_marginals(D, E, workspace=ws)
        Sd, So = call(); torch.cuda.synchronize()
        entry = {"n_states": nf + 1, "finite": bool(torch.isfinite(Sd).all() and torch.isfinite(So).all()),
                 "launches_marginals": _launches(call), "ms_marginals": _time(call, args.reps, args.warmup),
                 "ms_marginals_diag_only": _time(lambda: factor.chain_marginals(D, E, want_off=False, workspace=ws), args.reps, args.warmup)}
        rhs = torch.zeros((nf + 1, 15), dtype=torch.float64, device="cuda")
        entry["launches_solve"] = _launches(lambda: factor.chain_solve(D, E, rhs, workspace=ws))
        entry["ms_solve"] = _time(lambda: factor.chain_solve(D, E, rhs, workspace=ws), args.reps, args.warmup)
        out[name] = entry

    # the full sequence on the 5k chain: one LM step (eval -> blocks -> assemble -> solve -> retract), then the marginal covariances at
    # the new estimate (eval -> blocks -> assemble with lambda = 0 -> selected inversion)
    step = lambda: factor.chain_lm_step(1, dX, dR, dL)
    both = lambda: factor.chain_marginal_covariances(1, step()[0], dR, dL)
    out["chain_5k"]["launches_lm_step"] = _launches(step)
    out["chain_5k"]["ms_lm_step"] = _time(step, args.reps, args.warmup)
    out["chain_5k"]["launches_lm_step_plus_marginals"] = _launches(both)
    out["chain_5k"]["ms_lm_step_plus_marginals"] = _time(both, args.reps, args.warmup)
    torch.cuda.synchronize()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
