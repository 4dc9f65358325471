"""Cost of slod_update_basis against a full recomputation after a local change of the coefficient.

    python tools/update_bench.py --out update_bench.json [--reps 5] [--warmup 1] [--configs cfg4 2d]

Configurations: the default workload of bench.py (cfg 4: 3-D, 32^3 cells, n 2, l 2, uniform1e4) and its 2-D diffusion
workload (256^2 cells, n 2, l 2).  Change patterns on the bench's coefficient: one coarse cell at the centre, a block of
4^dim cells, and 1 % of the cells at seeded random positions.  For each pattern the two arms alternate in one process:
  update : slod_set_coefficient + slod_update_basis (basis and K)
  full   : slod_set_coefficient + slod_compute_basis + slod_assemble_coarse
each timed with the host clock around a device synchronise, after warm-up, median of --reps runs.  Between runs the
handle is brought back to the unchanged coefficient outside the timed region.  Writes one JSON line to --out with the
counts, the per-stage device times (slod_get_timings), launches, and the GPU name and power limit."""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
import bench  # noqa: E402

CONFIGS = {"cfg4": "diffusion3d_32c_l2_n2", "2d": "diffusion2d_256c_l2_n2"}
STAGES = ["solve", "dense", "select", "finish", "coarse"]


def patterns(w, seed=20261021):
    """name -> boolean [N]^dim mask (z, y, x) of the coarse cells whose table values change"""
    N, dim = 2 ** w["ref"], w["dim"]
    out = {}
    one = np.zeros((N,) * dim, dtype=bool)
    one[(N // 2,) * dim] = True
    out["one_cell"] = one
    blk = np.zeros((N,) * dim, dtype=bool)
    blk[tuple(slice(N // 2 - 2, N // 2 + 2) for _ in range(dim))] = True
    out[f"block_4^{dim}"] = blk
    rnd = np.zeros(N ** dim, dtype=bool)
    rnd[np.random.default_rng(seed).choice(N ** dim, size=max(1, N ** dim // 100), replace=False)] = True
    out["random_1pct"] = rnd.reshape((N,) * dim)
    return out


def changed_tables(w, tables, mask):
    """tables with every table cell inside a masked coarse cell multiplied by 1.5 (tables at least as fine as the cells)"""
    N, nl, dim = 2 ** w["ref"], 2 ** w["r"], w["dim"]
    k = nl // N
    big = mask
    for a in range(dim):
        big = np.repeat(big, k, axis=a)
    return [np.where(big.ravel(), t * 1.5, t) for t in tables]


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        power = None
    return name, power


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
        raise SystemExit("update_bench.py needs a CUDA device")
    pkg = importlib.import_module("dealii-slod_b200")
    name, power = gpu_info()
    result = {"tool": "update_bench", "gpu": name, "power_limit": power, "reps": args.reps, "warmup": args.warmup,
              "timing": "host clock around torch.cuda.synchronize(), median", "configs": {}}
    for cname in args.configs:
        wname = CONFIGS[cname]
        w = bench.WORKLOADS[wname]
        base = bench.make_tables(w)
        ctx = pkg.SlodContext(dim=w["dim"], spacedim=w["s"], n_global_refinements=w["ref"], n_subdivisions=w["n"],
                              oversampling=w["ell"], stabilize=True, problem=0 if w["s"] == 1 else 1, device=0)

        def set_tables(ts):
            for f, t in enumerate(ts):
                ctx.set_coefficient(f, w["r"], t)

        def full(ts):
            set_tables(ts)
            ctx.compute_basis()
            ctx.assemble_coarse()
            torch.cuda.synchronize()

        def update(ts):
            set_tables(ts)
            counts = ctx.update_basis()
            torch.cuda.synchronize()
            return counts

        full(base)
        cres = {"workload": wname, "config": bench.config_of(w, wname), "patterns": {}}
        for pname, mask in patterns(w).items():
            changed = changed_tables(w, base, mask)
            arms = {"update": [], "full": []}
            stage = {"update": [], "full": []}
            launches = {}
            counts = None
            for rep in range(args.warmup + args.reps):
                for arm in ("update", "full"):
                    l0 = ctx.launch_count
                    t0 = time.perf_counter()
                    if arm == "update":
                        counts = update(changed)
                    else:
                        full(changed)
                    dt = time.perf_counter() - t0
                    tm = ctx.timings()
                    launches[arm] = ctx.launch_count - l0
                    if rep >= args.warmup:
                        arms[arm].append(dt * 1e3)
                        stage[arm].append(tm[:5])
                    if arm == "update":
                        update(base)       # back to the unchanged coefficient (and its baseline), untimed
                    else:
                        full(base)
            med = {a: float(np.median(v)) for a, v in arms.items()}
            cres["patterns"][pname] = {
                "cells_changed": int(mask.sum()), "patches_recomputed": counts["patches"],
                "row_blocks_recomputed": counts["row_blocks"], "n_patches": ctx.n_patches,
                "update_ms": med["update"], "full_ms": med["full"], "speedup": med["full"] / med["update"],
                "update_ms_runs": arms["update"], "full_ms_runs": arms["full"],
                "stage_ms_update": dict(zip(STAGES, np.median(stage["update"], axis=0).tolist())),
                "stage_ms_full": dict(zip(STAGES, np.median(stage["full"], axis=0).tolist())),
                "launches": launches}
            print(cname, pname, json.dumps(cres["patterns"][pname]), flush=True)
        result["configs"][cname] = cres
        ctx.close()
        del ctx
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(result) + "\n")
    print(json.dumps(result))


if __name__ == "__main__":
    main()
