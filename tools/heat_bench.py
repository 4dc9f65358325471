"""Coarse mass matrix and theta-scheme time stepping on the SLOD space at the headline workload.

    python tools/heat_bench.py [--out profiles/heat_bench.json] [--workload NAME] [--steps 20] [--k 16] [--dt 1e-3]
                               [--reps 3]

Builds the workload of bench.py (default: the headline 3-D workload, 32^3 cells, oversampling 2), runs the offline phase
once, then times, after one warm-up call of each, the median over --reps repetitions of:
  * slod_assemble_coarse_mass: host clock around the (synchronising) call, and the CUDA-event times of its two kernels
    (M_h phi and the product C^T (M_h C), slod_get_timings [6] / [7]);
  * slod_heat_solve: --steps backward-Euler steps for the forcing f = 1 from u0 = 0, host clock, CG steps per time step;
  * slod_heat_solve_batch with --k seeded random forcings, the same steps: host clock, CG steps per time step (the
    largest over the columns, which sets the group's step count);
  * slod_heat_theta_solve at theta = 1/2 (Crank-Nicolson) for the same forcing with g = sin(pi t / T), T = steps dt,
    without and with two Rannacher start-up steps, and with 8 fields (f = 1 and 7 seeded ones, seeded g);
  * slod_heat_theta_solve_batch at theta = 1/2 for the --k forcings (one field each, g as above) and with 8 fields per
    column (seeded);
  * both at theta = 1/2 with per-step forcing: steps + 1 seeded fields and g the identity (every step reads all
    steps + 1 coarse loads, so this time grows with the number of steps).
All CG solves stop at a reduction of 1e-10.  Host-buffer copies are included in the host times.  The device name and
power limit are read in the same run.  Writes one JSON line to --out and prints it.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

pkg = importlib.import_module("dealii-slod_b200")
CG = dict(max_steps=20000, tolerance=0.0, reduction=1e-10)


def _device():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        power = q[0].split(",")[-1].strip() if q else None
    except (OSError, subprocess.SubprocessError):
        power = None
    return name, power


def _median_ms(fn, reps):
    fn()   # warm-up
    ts, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "heat_bench.json"))
    ap.add_argument("--workload", default=bench.DEFAULT_WORKLOAD, choices=sorted(bench.WORKLOADS))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--dt", type=float, default=1e-3)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("heat_bench.py needs a CUDA device (no CPU fallback)")
    w = bench.WORKLOADS[args.workload]
    ctx = pkg.SlodContext(dim=w["dim"], spacedim=w["s"], n_global_refinements=w["ref"], n_subdivisions=w["n"],
                          oversampling=w["ell"], stabilize=True, problem=0 if w["s"] == 1 else 1)
    for f, t in enumerate(bench.make_tables(w)):
        ctx.set_coefficient(f, w["r"], t)
    ctx.compute_basis()
    ctx.assemble_coarse()
    nf, nc = ctx.n_fine, ctx.n_patches * ctx.s

    ev = []

    def mass():
        ctx.assemble_coarse_mass()
        ev.append(ctx.timings()[6:8].copy())
    mass_ms, _ = _median_ms(mass, args.reps)
    ev = np.array(ev[1:])
    h = 1.0 / (2 ** w["ref"] * w["n"])
    f1 = np.full(nf, h ** w["dim"])   # f = 1: the load vector of the interior nodes
    single_ms, (_, st1) = _median_ms(lambda: ctx.heat_solve(f1, None, args.dt, args.steps, args.steps, **CG), args.reps)
    rng = np.random.default_rng(17)
    F = rng.standard_normal((args.k, nf)) * h ** w["dim"]
    batch_ms, (_, stk) = _median_ms(lambda: ctx.heat_solve_batch(F, None, args.dt, args.steps, args.steps, **CG),
                                    args.reps)
    T = args.dt * args.steps
    g1 = np.sin(np.pi * np.arange(args.steps + 1) * args.dt / T)[:, None]
    nq = 8
    F8 = np.concatenate([f1[None], rng.standard_normal((nq - 1, nf)) * h ** w["dim"]])
    G8 = rng.standard_normal((args.steps + 1, nq))
    theta = {}
    FP = rng.standard_normal((args.steps + 1, nf)) * h ** w["dim"]
    GP = np.eye(args.steps + 1)
    for key, fields, g, ns in (("cn", f1[None], g1, 0), ("cn_startup2", f1[None], g1, 2), ("cn_fields8", F8, G8, 0),
                               ("cn_per_step", FP, GP, 0)):
        ms, (_, st) = _median_ms(lambda: ctx.heat_theta_solve(fields, g, None, 0.5, args.dt, args.steps, args.steps,
                                                              n_startup=ns, **CG), args.reps)
        theta[key] = {"n_fields": fields.shape[0], "n_startup": ns, "ms": ms, "ms_per_step": ms / args.steps,
                      "cg_steps": st.tolist(), "ms_per_cg_step": ms / max(int(st.sum()), 1)}
    Gk = np.broadcast_to(g1, (args.k,) + g1.shape)
    FK8 = rng.standard_normal((args.k, nq, nf)) * h ** w["dim"]
    GK8 = rng.standard_normal((args.k, args.steps + 1, nq))
    FKP = np.broadcast_to(FP, (args.k,) + FP.shape)
    GKP = np.broadcast_to(GP, (args.k,) + GP.shape)
    for key, fields, g in (("cn_batch", F[:, None], Gk), ("cn_batch_fields8", FK8, GK8),
                           ("cn_batch_per_step", FKP, GKP)):
        ms, (_, st) = _median_ms(lambda: ctx.heat_theta_solve_batch(fields, g, None, 0.5, args.dt, args.steps,
                                                                    args.steps, **CG), args.reps)
        theta[key] = {"k": args.k, "n_fields": fields.shape[1], "ms": ms, "ms_per_step": ms / args.steps,
                      "ms_per_step_per_rhs": ms / args.steps / args.k, "cg_steps_max": st.max(axis=1).tolist(),
                      "ms_per_cg_step": ms / max(int(st.max(axis=1).sum()), 1)}
    name, power = _device()
    row = {
        "metric": "heat", "workload": args.workload, "device": name, "power_limit": power,
        "n_fine": nf, "n_coarse": nc, "reps": args.reps, "dt": args.dt, "time_steps": args.steps, "cg": CG,
        "timing": "median of host clocks around synchronising C-ABI calls (host-buffer copies included); kernel times "
                  "from CUDA events",
        "assemble_coarse_mass_ms": mass_ms,
        "mass_apply_event_ms": float(np.median(ev[:, 0])), "mass_product_event_ms": float(np.median(ev[:, 1])),
        "mass_apply_bytes": 2 * 8 * nc * ctx.basis_stride,   # phi read once, M_h phi written once
        "heat_solve": {"ms": single_ms, "ms_per_step": single_ms / args.steps, "cg_steps": st1.tolist(),
                       "ms_per_cg_step": single_ms / max(int(st1.sum()), 1)},
        "heat_solve_batch": {"k": args.k, "ms": batch_ms, "ms_per_step": batch_ms / args.steps,
                             "ms_per_step_per_rhs": batch_ms / args.steps / args.k,
                             "cg_steps_max": stk.max(axis=1).tolist(),
                             "ms_per_cg_step": batch_ms / max(int(stk.max(axis=1).sum()), 1)},
        "heat_theta_solve": theta,
    }
    line = json.dumps(row)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
