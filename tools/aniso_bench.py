"""Offline phase with an anisotropic coefficient (SLOD_PROBLEM_DIFFUSION_TENSOR) against the scalar problem.

    python tools/aniso_bench.py --out profiles/aniso_bench.json [--reps 5] [--warmup 1] [--configs cfg4 2d]

Configurations: bench.py's cfg 4 (3-D, 32^3 cells, n 2, l 2) and the 2-D workload of tools/update_bench.py (256^2
cells, n 2, l 2).  Three coefficients on one geometry, alternating in one process:
  scalar    : the bench's alpha through slod_set_coefficient
  iso       : the tensor alpha I with the same alpha
  laminate  : a rotated laminate (tools/aniso_oracle.py) whose across-layer conductivity is the same alpha field's
              max / min contrast
Each arm is timed as slod_compute_basis + slod_assemble_coarse with the host clock around a device synchronise, after
warm-up, median of --reps runs.  Recorded per arm: the time, the per-stage device times (slod_get_timings), the kernel
plan (slod_get_plan), the histogram of selection paths (slod_get_patch_diagnostics [5]: 0 LOD, 1 Cholesky fast path,
2 Jacobi, 3 QL), the summed QL iterations / Jacobi sweeps ([6]) and the GPU name and power limit.  With the split
solver the solve stage is also split into its factor kernel and the triangular solves."""
import argparse
import importlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True
import bench  # noqa: E402
from aniso_oracle import laminate  # noqa: E402
from update_bench import CONFIGS, STAGES, gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--configs", nargs="+", default=list(CONFIGS), choices=list(CONFIGS))
    args = ap.parse_args()
    if args.reps < 5:
        ap.error("--reps must be at least 5 (the median of at least 5 runs is reported)")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("aniso_bench.py needs a CUDA device")
    pkg = importlib.import_module("dealii-slod_b200")
    name, power = gpu_info()
    result = {"tool": "aniso_bench", "gpu": name, "power_limit": power, "reps": args.reps, "warmup": args.warmup,
              "timing": "host clock around torch.cuda.synchronize(), median", "configs": {}}
    for cname in args.configs:
        wname = CONFIGS[cname]
        w = bench.WORKLOADS[wname]
        dim, r = w["dim"], w["r"]
        alpha = bench.make_tables(w)[0]
        iso = np.zeros((alpha.size, dim * (dim + 1) // 2))
        iso[:, :dim] = alpha[:, None]
        lam = laminate(dim, r, contrast=float(alpha.max() / alpha.min()))
        ctxs = {}
        for arm in ("scalar", "iso", "laminate"):
            c = pkg.SlodContext(dim=dim, spacedim=1, n_global_refinements=w["ref"], n_subdivisions=w["n"],
                                oversampling=w["ell"], stabilize=True,
                                problem=pkg.PROBLEM_DIFFUSION if arm == "scalar" else pkg.PROBLEM_DIFFUSION_TENSOR,
                                device=0)
            if arm == "scalar":
                c.set_coefficient(0, r, alpha)
            else:
                c.set_coefficient_tensor(r, iso if arm == "iso" else lam)
            ctxs[arm] = c
        times = {a: [] for a in ctxs}
        stages = {a: [] for a in ctxs}
        for rep in range(args.warmup + args.reps):
            for arm, c in ctxs.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                c.compute_basis()
                c.assemble_coarse()
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                if rep >= args.warmup:
                    times[arm].append(dt * 1e3)
                    stages[arm].append(c.timings()[:6])
        cres = {"workload": wname, "config": bench.config_of(w, wname), "arms": {}}
        for arm, c in ctxs.items():
            paths = np.zeros(4, dtype=int)
            eig_iters = 0
            for pid in range(c.n_patches):
                dg = c.diagnostics(pid)
                paths[int(dg[5])] += 1
                eig_iters += int(dg[6])
            st = np.median(stages[arm], axis=0)
            stage_ms = dict(zip(STAGES, st[:5].tolist()))
            if st[5] > 0:   # split solver: its factor kernel and the triangular solves (one chunk)
                stage_ms["factor"], stage_ms["trisolve"] = float(st[5]), float(st[0] - st[5])
            cres["arms"][arm] = {
                "ms": float(np.median(times[arm])), "ms_runs": times[arm], "stage_ms": stage_ms,
                "eigen_iterations": eig_iters,
                "plan": c.plan(), "selection_paths": dict(zip(["lod", "cholesky", "jacobi", "ql"], paths.tolist()))}
            print(cname, arm, json.dumps(cres["arms"][arm]), flush=True)
        result["configs"][cname] = cres
        for c in ctxs.values():
            c.close()
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(result) + "\n")
    print(json.dumps(result))


if __name__ == "__main__":
    main()
