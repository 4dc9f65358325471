"""Batched online phase against k single-vector calls: C^T F, coarse CG and C U for k right-hand sides.

    python tools/online_batch_bench.py --out DIR [--workload NAME] [--ks 1,4,16,32] [--reps 5] [--profile]

Builds the workload of bench.py (default: the headline 3-D workload), runs the offline phase once, then for every k
and seeded random forcings times, with host clocks around the (synchronising) C-ABI calls, after a warm-up of every
shape, the median over --reps repetitions of: the batched C^T F, the batched CG (tolerance 0, reduction 1e-10), the
batched C U, and the loop of k single-vector calls doing the same work.  It also records CUDA-event time per CG step of
the batched solve and the K bytes streamed per step over that time, and checks that batch and single results agree.
The batched outputs reuse their page-locked blocks between repetitions (reuse=True): no host allocation is timed.
Prints one JSON line and writes it (and, with --profile, a kernel table of one k = 16 chain) under --out only.
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


def _timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return time.perf_counter() - t0, out


def _rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for the JSON line (and the profile)")
    ap.add_argument("--workload", default=bench.DEFAULT_WORKLOAD, choices=sorted(bench.WORKLOADS))
    ap.add_argument("--ks", default="1,4,16,32")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--profile", action="store_true", help="torch.profiler kernel table of one k = 16 chain")
    args = ap.parse_args()
    if args.reps < 5:
        ap.error("--reps must be at least 5")
    ks = [int(x) for x in args.ks.split(",")]
    os.makedirs(args.out, exist_ok=True)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement runs on the GPU only")
    name, power = _device()

    w = bench.WORKLOADS[args.workload]
    ctx = pkg.SlodContext(dim=w["dim"], spacedim=w["s"], n_global_refinements=w["ref"], n_subdivisions=w["n"],
                          oversampling=w["ell"], stabilize=True, problem=0 if w["s"] == 1 else 1)
    for f, t in enumerate(bench.make_tables(w)):
        ctx.set_coefficient(f, w["r"], t)
    ctx.compute_basis()
    ctx.assemble_coarse()
    nf, nc = ctx.n_fine, ctx.n_patches * ctx.s
    k_bytes = 8 * nc * ctx.ell_width   # the block-ELL K, read once per CG step whatever k is
    rng = np.random.default_rng(2024)

    rows = []
    for k in ks:
        F = rng.standard_normal((k, nf))
        # warm-up of every shape
        B = ctx.coarse_rhs_batch(F, reuse=True)
        U, steps, _ = ctx.coarse_solve_batch(B, reuse=True, **CG)
        ctx.prolongate_batch(U, reuse=True)
        b1 = ctx.coarse_rhs(F[0])
        ctx.prolongate(ctx.coarse_solve(b1, **CG)[0])
        t = {key: [] for key in ("rhs", "cg", "prolong", "rhs1", "cg1", "prolong1", "cg_event")}
        for _ in range(args.reps):
            dt, B = _timed(lambda: ctx.coarse_rhs_batch(F, reuse=True))
            t["rhs"].append(dt)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            dt, (U, steps, res) = _timed(lambda: ctx.coarse_solve_batch(B, reuse=True, **CG))
            e1.record()
            e1.synchronize()
            t["cg"].append(dt)
            t["cg_event"].append(e0.elapsed_time(e1) * 1e-3)
            dt, Uf = _timed(lambda: ctx.prolongate_batch(U, reuse=True))
            t["prolong"].append(dt)
            a = b = c = 0.0
            singles = []
            for j in range(k):
                d1, bj = _timed(lambda: ctx.coarse_rhs(F[j]))
                d2, (uj, sj, _) = _timed(lambda: ctx.coarse_solve(bj, **CG))
                d3, ufj = _timed(lambda: ctx.prolongate(uj))
                a, b, c = a + d1, b + d2, c + d3
                singles.append((bj, uj, sj, ufj))
            t["rhs1"].append(a)
            t["cg1"].append(b)
            t["prolong1"].append(c)
        med = {key: float(np.median(v)) * 1e3 for key, v in t.items()}
        rhs_err = max(_rel(B[j], s[0]) for j, s in enumerate(singles))
        u_err = max(float(np.linalg.norm(U[j] - s[1]) / np.linalg.norm(s[1])) for j, s in enumerate(singles))
        uf_err = max(_rel(Uf[j], ctx.prolongate(s[1])) for j, s in enumerate(singles))
        step_diff = max(abs(int(steps[j]) - s[2]) for j, s in enumerate(singles))
        n_steps = int(steps.max())
        chain = med["rhs"] + med["cg"] + med["prolong"]
        chain1 = med["rhs1"] + med["cg1"] + med["prolong1"]
        rows.append({
            "k": k, "batch_ms": {"rhs": med["rhs"], "cg": med["cg"], "prolongate": med["prolong"], "chain": chain},
            "single_loop_ms": {"rhs": med["rhs1"], "cg": med["cg1"], "prolongate": med["prolong1"], "chain": chain1},
            "per_rhs_ms": {"batch": chain / k, "single": chain1 / k}, "throughput_ratio": chain1 / chain,
            "cg_steps_max": n_steps, "cg_event_ms_per_step": med["cg_event"] / n_steps,
            "K_bytes_per_step": k_bytes, "K_TB_per_s": k_bytes / (med["cg_event"] * 1e-3 / n_steps) / 1e12,
            "agree": {"rhs_rel": rhs_err, "u_rel": u_err, "u_fine_rel": uf_err, "steps_diff": step_diff,
                      "ok": rhs_err <= 1e-12 and uf_err <= 1e-9 and u_err <= 1e-9 and step_diff <= 1},
        })
        print(json.dumps({"k": k, "chain_ms": chain, "single_chain_ms": chain1, "ratio": chain1 / chain}),
              file=sys.stderr)

    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        F = rng.standard_normal((16, nf))
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            B = ctx.coarse_rhs_batch(F, reuse=True)
            U, _, _ = ctx.coarse_solve_batch(B, reuse=True, **CG)
            ctx.prolongate_batch(U, reuse=True)
        with open(os.path.join(args.out, "online_batch_profile_k16.txt"), "w") as fh:
            fh.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=30))

    line = {"metric": "online_batch", "workload": args.workload, "device": name, "power_limit": power,
            "n_fine": nf, "n_coarse": nc, "reps": args.reps, "timing": "median of host clocks around synchronising "
            "C-ABI calls (host-buffer copies included)", "cg": CG, "rows": rows}
    txt = json.dumps(line)
    with open(os.path.join(args.out, "online_batch_bench.json"), "w") as fh:
        fh.write(txt + "\n")
    print(txt)
    ctx.close()


if __name__ == "__main__":
    main()
