"""Newmark time stepping of the wave equation on the SLOD space at the headline workload.

    python tools/wave_bench.py [--out profiles/wave_bench.json] [--workload NAME] [--steps 20] [--k 16] [--dt 1e-3]
                               [--reps 5]

Builds the workload of bench.py (default: the headline 3-D workload, 32^3 cells, oversampling 2), runs the offline phase,
slod_assemble_coarse and slod_assemble_coarse_mass once, then times, after one warm-up call of each, the median over
--reps repetitions of (host clock around the synchronising C-ABI call, host-buffer copies included):
  * slod_wave_solve at beta = 1/4 (average acceleration), --steps steps of --dt from seeded u0, v0, no forcing;
  * slod_wave_solve_batch at beta = 1/4 for --k seeded columns, the same steps;
  * both at beta = 0 (central differences) at 0.9 x the stable step 2 / sqrt(lambda_max(M_H^-1 K)), lambda_max from a
    power iteration on the host CSR copies of K and M_H (scipy CG for the M_H solves).
Each run records ms per step, CG steps per step (the largest over the columns for the batch) and the largest relative
change of the energy 1/2 v^T M_H v + 1/2 u^T K u over the trajectory (energy_out at every step).  All CG solves stop
at a reduction of 1e-10.  The device name and power limit are read in the same run.  Writes one JSON line to --out and
prints it.
"""
import argparse
import importlib
import json
import os
import sys

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from heat_bench import _device, _median_ms  # noqa: E402

pkg = importlib.import_module("dealii-slod_b200")
CG = dict(max_steps=20000, tolerance=0.0, reduction=1e-10)


def _csr(t, n):
    rowptr, col, val = t
    return sp.csr_matrix((val.copy(), col.copy(), rowptr.copy()), shape=(n, n))


def lambda_max(K, M, iters=40, seed=3):
    """Power iteration for the largest eigenvalue of M^-1 K (Rayleigh quotient x^T K x / x^T M x, which approaches it
    from below), until it changes by less than 1e-6 relative; returns (lambda, iterations, last relative change)."""
    x = np.random.default_rng(seed).standard_normal(K.shape[0])
    lam, change = 0.0, 1.0
    for it in range(1, iters + 1):
        y, info = spla.cg(M, K @ x, rtol=1e-8, maxiter=1000)
        if info != 0:
            raise RuntimeError(f"scipy CG on M_H did not converge ({info})")
        x = y / np.linalg.norm(y)
        new = float(x @ (K @ x)) / float(x @ (M @ x))
        change = abs(new - lam) / new
        lam = new
        print(f"power iteration {it}: lambda {lam:.9g}, change {change:.2e}", flush=True)
        if change <= 1e-6:
            break
    return lam, it, change


def _run(beta, dt, steps, U0, V0, ctx, reps):
    if U0.ndim == 1:
        ms, (_, _, E, st) = _median_ms(lambda: ctx.wave_solve(None, None, U0, V0, beta, dt, steps, 1, **CG), reps)
        cg, drift = st[1:], float(np.abs(E / E[0] - 1.0).max())
        return {"beta": beta, "dt": dt, "k": 1, "ms": ms, "ms_per_step": ms / steps,
                "cg_steps_start": int(st[0]), "cg_steps_per_step": float(cg.mean()), "energy_drift": drift}
    ms, (_, _, E, st) = _median_ms(lambda: ctx.wave_solve_batch(None, None, U0, V0, beta, dt, steps, 1, **CG), reps)
    k = U0.shape[0]
    cg, drift = st[1:].max(axis=1), float(np.abs(E / E[0] - 1.0).max())
    return {"beta": beta, "dt": dt, "k": k, "ms": ms, "ms_per_step": ms / steps, "ms_per_step_per_rhs": ms / steps / k,
            "cg_steps_start": int(st[0].max()), "cg_steps_per_step": float(cg.mean()), "energy_drift": drift}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "wave_bench.json"))
    ap.add_argument("--workload", default=bench.DEFAULT_WORKLOAD, choices=sorted(bench.WORKLOADS))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--dt", type=float, default=1e-3)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("wave_bench.py needs a CUDA device (no CPU fallback)")
    w = bench.WORKLOADS[args.workload]
    ctx = pkg.SlodContext(dim=w["dim"], spacedim=w["s"], n_global_refinements=w["ref"], n_subdivisions=w["n"],
                          oversampling=w["ell"], stabilize=True, problem=0 if w["s"] == 1 else 1)
    for f, t in enumerate(bench.make_tables(w)):
        ctx.set_coefficient(f, w["r"], t)
    ctx.compute_basis()
    ctx.assemble_coarse()
    ctx.assemble_coarse_mass()
    nc = ctx.n_patches * ctx.s
    lam, lam_iters, lam_change = lambda_max(_csr(ctx.coarse_csr(), nc), _csr(ctx.coarse_mass_csr(), nc))
    dt_explicit = 0.9 * 2.0 / np.sqrt(lam)
    rng = np.random.default_rng(17)
    U0, V0 = rng.standard_normal((args.k, nc)), rng.standard_normal((args.k, nc))
    runs = {}
    for key, beta, dt in (("average_acceleration", 0.25, args.dt), ("central_difference", 0.0, dt_explicit)):
        runs[key] = _run(beta, dt, args.steps, U0[0], V0[0], ctx, args.reps)
        runs[key + "_batch"] = _run(beta, dt, args.steps, U0, V0, ctx, args.reps)
    name, power = _device()
    row = {
        "metric": "wave", "workload": args.workload, "device": name, "power_limit": power,
        "n_coarse": nc, "reps": args.reps, "time_steps": args.steps, "cg": CG,
        "lambda_max": lam, "lambda_max_power_iterations": lam_iters, "lambda_max_last_change": lam_change,
        "explicit_dt": dt_explicit,
        "timing": "median of host clocks around synchronising C-ABI calls (host-buffer copies included; energy_out at "
                  "every step)",
        "runs": runs,
    }
    line = json.dumps(row)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
