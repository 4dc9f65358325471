#!/usr/bin/env python
"""Benchmark of the SLOD offline phase (BASELINE.json metric: SLOD basis patches/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over the whole synthetic problem: per-patch basis computation
(source/LOD.cc:296-768) for every patch, then the coarse stiffness matrix (source/LOD.cc:860-973).
Default workload: the configuration the metric is quoted on -- 3-D diffusion, 32^3 = 2^15 coarse cells,
oversampling 2, 2 subdivisions, uniform random coefficient in [1, 1e4] on the fine sub-cell grid (SURVEY 8d,
cfg 4a/5).  N > 1 (torchrun): contiguous Morton ranges of patches per rank, one NCCL all-gather of A*phi before
the coarse matrix and one of the K row blocks after it; timing = max over ranks of CUDA-event time.

value : patches/s with the coefficient already resident in HBM (device-buffer entry points).
e2e   : the same through the host-buffer C ABI (slod_set_coefficient -> slod_compute_basis ->
        slod_assemble_coarse -> slod_get_coarse_csr + slod_get_all_basis), host<->device copies inside the timed region.

--dump-outputs DIR writes what the timed path computed in its last step (see dump_outputs) so that two builds can be
compared output for output on identical, seeded inputs.

bench.py writes nothing into the repository (it may be read-only): it runs the libraries that __graft_entry__.build()
left in the tree, so rebuild after changing the CUDA sources.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True   # before the project's modules are imported: no __pycache__ in the repository
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: dim, s, ref, n, ell, r, kind, seed
    "diffusion3d_32c_l2_n2": dict(dim=3, s=1, ref=5, n=2, ell=2, r=6, kind="uniform1e4", seed=3001),
    "diffusion3d_16c_l2_n2": dict(dim=3, s=1, ref=4, n=2, ell=2, r=5, kind="uniform1e4", seed=3001),
    "diffusion2d_256c_l2_n2": dict(dim=2, s=1, ref=8, n=2, ell=2, r=8, kind="uniform100", seed=1234),
    "elasticity2d_128c_l1_n2": dict(dim=2, s=2, ref=7, n=2, ell=1, r=6, kind="uniform100", seed=2001),
    "diffusion2d_16c_l2_n2": dict(dim=2, s=1, ref=4, n=2, ell=2, r=5, kind="uniform100", seed=1234),
}
DEFAULT_WORKLOAD = "diffusion3d_32c_l2_n2"
FP64_PEAK_FALLBACK = 37.2   # only if the in-run probe fails: measured earlier on this pool's B200 (mma.sync m8n8k4 f64; DFMA 36.3)


def make_tables(w):
    rs = np.random.default_rng(w["seed"])
    n = (2 ** w["r"]) ** w["dim"]
    out = []
    for f in range(1 if w["s"] == 1 else 2):
        u = rs.random(n)
        hi = 1e4 if w["kind"] == "uniform1e4" else 100.0
        out.append(1.0 + (hi - 1.0) * u)
    return out


def patch_shapes(w):
    """Per patch: Ni, bw, Ncd, Nb (vectorised closed forms of slod::make_geom)."""
    dim, s, ref, n, ell = w["dim"], w["s"], w["ref"], w["n"], w["ell"]
    N = 2 ** ref
    c = np.arange(N)
    lo = np.maximum(c - ell, 0)
    hi = np.minimum(c + ell, N - 1)
    m1 = hi - lo + 1
    dl = (lo == 0).astype(int)
    dh = (hi == N - 1).astype(int)
    grids = np.meshgrid(*([np.arange(N)] * dim), indexing="ij")
    m = [m1[g].ravel() for g in grids]
    nob = [(m1 * n + 1 - (1 - dl) - (1 - dh))[g].ravel() for g in grids]
    p = [mm * n + 1 for mm in m]
    q = [pp - 2 for pp in p]
    Ni = s * np.prod(q, axis=0)
    Ncd = s * np.prod(m, axis=0)
    nnodes = np.prod(p, axis=0)
    Nb = s * (nnodes - np.prod(nob, axis=0))
    nbw = (q[0] * q[1] + q[0] + 1) if dim == 3 else (q[0] + 1)
    bw = np.minimum(s * nbw + s - 1, Ni - 1)
    return dict(Ni=Ni.astype(float), bw=bw.astype(float), Ncd=Ncd.astype(float), Nb=Nb.astype(float),
                Nf=(s * nnodes).astype(float))


def flop_model(w):
    """Algorithmic flops per kernel, summed over all patches (banded-solver model of SURVEY 8d)."""
    sh = patch_shapes(w)
    Ni, bw, Ncd, Nb, Nf = sh["Ni"], sh["bw"], sh["Ncd"], sh["Nb"], sh["Nf"]
    st = 27.0 if w["dim"] == 3 else 9.0
    s = w["s"]
    solve = Ni * bw * bw + 4.0 * Ni * bw * Ncd
    dense = 2.0 * Ncd ** 3 + 2.0 * Nb * st * s * Ncd + 2.0 * Nb * Ncd ** 2 + 2.0 * Nb * Ncd ** 2
    select = s * 12.0 * (Ncd - 1) ** 3
    finish = s * (2.0 * Ni * Ncd + 2.0 * Nf * st * s)
    return dict(patch_solve=float(solve.sum()), patch_dense=float(dense.sum()), patch_select=float(select.sum()),
                patch_finish=float(finish.sum()))


class ClockSampler:
    def __init__(self, index=0):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, args=(index,), daemon=True)

    def _run(self, index):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(index), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for nm, v in zip(names, out[2:]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the C++ restatement of the reference algorithm on the host cores
# ------------------------------------------------------------------------------------------------------
def cpu_sample_ids(w, block):
    """One Morton-contiguous block of 1 / 2^dim of the patches (an octant of the 32^3 mesh = 4096 patches at cfg 4):
    the same mix of interior / face / edge / corner patches as the whole mesh, and a compact set whose coarse-matrix
    rows mostly stay inside the block."""
    n = n_total(w)
    nb = 2 ** w["dim"]
    size = max(1, n // nb)
    b = block % nb
    return np.arange(b * size, min(n, (b + 1) * size), dtype=np.int64)


def cpu_port_step(w, tables, block):
    """One bounded sample of the offline phase on the host cores, through the C-ABI of the C++ port
    (oracle/cpu/slod_cpu.cc, all hardware threads): handle set-up, coefficient upload, every stage of
    LOD::compute_basis_function_candidates (source/LOD.cc:296-768) for the patches of one block, and the rows of
    LOD::assemble_global_matrix (source/LOD.cc:860-973) of those patches (columns inside the block).
    Returns (patches/s, seconds, handle, ids)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from cpu_port import CpuSlod
    ids = cpu_sample_ids(w, block)
    t0 = time.perf_counter()
    cpu = CpuSlod(dim=w["dim"], spacedim=w["s"], n_global_refinements=w["ref"], n_subdivisions=w["n"],
                  oversampling=w["ell"], stabilize=True, problem=0 if w["s"] == 1 else 1)
    for f, t in enumerate(tables):
        cpu.set_coefficient(f, w["r"], t)
    cpu.compute_patches(ids)
    cpu.assemble_coarse_subset()
    dt = time.perf_counter() - t0
    return ids.size / dt, dt, cpu, ids


def cpu_sample_text(w, n_ids, cores):
    return (f"{n_ids} patches per step = one Morton-contiguous 1/{2 ** w['dim']} block of the {n_total(w)} patches "
            f"(block index rotates with the step); C++ restatement of source/LOD.cc:296-768 + :860-973 "
            f"(oracle/cpu/slod_cpu.cc: banded Cholesky, Householder+QL eigen-solver, std::thread over patches, {cores} "
            "threads), timed region = handle set-up + coefficient upload + basis + coarse-matrix rows of the block; "
            "the deal.II/Trilinos reference itself cannot be built in this image")


def run_reference(args, w, wname):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    tables = make_tables(w)
    rates = []
    cores = os.cpu_count() or 1
    n_ids = 0
    for it in range(args.warmup + args.steps):
        rate, dt, cpu, ids = cpu_port_step(w, tables, it)
        cores, n_ids = cpu.threads, ids.size
        cpu.close()
        if it >= args.warmup:
            rates.append((rate, dt))
    value = float(np.mean([r for r, _ in rates]))
    ms = float(np.mean([d for _, d in rates]) * 1e3)
    line = {
        "impl": "reference", "metric": "slod_basis_patches_per_s", "value": value, "unit": "patches/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_of(w, wname),
        "cpu_baseline": {"value": value, "unit": "patches/s", "cores": cores, "kind": "port", "language": "c++",
                         "sample": cpu_sample_text(w, n_ids, cores)},
        "e2e": {"value": value, "unit": "patches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def parity_against_cpu(w, cpu, ids, phi_dev, aphi_dev, gpu_csr, diag_of):
    """GPU results against the C++ CPU port on the sample of the CPU baseline (outside every timed region):
    per-patch ||phi_gpu - phi_cpu||_2 (both have unit norm), the same for A phi relative to ||A phi||, truncation step
    counts, and the coarse-matrix entries of the sample rows on the sample columns relative to max |K|."""
    import scipy.sparse as sp
    s = w["s"]
    errs, aerrs, steps_bad, interior = [], [], 0, []
    N, ell = 2 ** w["ref"], w["ell"]
    for pid in ids:
        pid = int(pid)
        nf = cpu.patch_info(pid)["n_fine"]
        c = [0] * w["dim"]
        for b in range(w["ref"]):
            for a in range(w["dim"]):
                c[a] |= ((pid >> (w["dim"] * b + a)) & 1) << b
        interior.append(all(ell <= x <= N - 1 - ell for x in c))
        for d in range(s):
            pc, ac = cpu.basis(pid, d)
            pg = phi_dev[pid, d, :nf].cpu().numpy()
            ag = aphi_dev[pid, d, :nf].cpu().numpy()
            errs.append(float(np.linalg.norm(pg - pc)))
            aerrs.append(float(np.linalg.norm(ag - ac) / np.linalg.norm(ac)))
            steps_bad += int(cpu.diagnostics(pid, d)[1]) != int(diag_of(pid, d)[1])
    errs, aerrs = np.array(errs), np.array(aerrs)
    interior = np.repeat(np.array(interior), s)
    out = {"against": "oracle/cpu/slod_cpu.cc (C++ CPU port) on the cpu_baseline sample", "n_patches": int(len(ids)),
           "phi_max": float(errs.max()), "phi_p99": float(np.quantile(errs, 0.99)), "phi_median": float(np.median(errs)),
           "phi_frac_le_1e-10": float((errs <= 1e-10).mean()),
           "phi_max_full_size_patches": float(errs[interior].max()) if interior.any() else None,
           "n_full_size_patches": int(interior.sum()),
           "aphi_rel_max": float(aerrs.max()), "truncation_step_mismatches": int(steps_bad)}
    if gpu_csr is not None:
        rowptr, col, val = gpu_csr
        n = rowptr.size - 1
        Kg = sp.csr_matrix((val, col, rowptr), shape=(n, n))
        rp, cc, vv = cpu.coarse_csr()
        Kc = sp.csr_matrix((vv, cc, rp), shape=(n, n))
        rows = (np.asarray(ids)[:, None] * s + np.arange(s)[None, :]).ravel()
        sub_g = Kg[rows][:, rows]
        sub_c = Kc[rows][:, rows]
        kmax = float(np.abs(val).max())
        out["K_rel_max"] = float(np.abs((sub_g - sub_c)).max() / kmax)
        out["K_entries_compared"] = int(sub_c.nnz)
    return out


def n_total(w):
    return (2 ** w["ref"]) ** w["dim"]


def config_of(w, wname):
    return {"workload": wname, "dim": w["dim"], "spacedim": w["s"], "coarse_cells_per_axis": 2 ** w["ref"],
            "n_patches": n_total(w), "oversampling": w["ell"], "n_subdivisions": w["n"], "stabilize": True,
            "coefficient": f"{w['kind']} on 2^{w['r']} cells/axis, PCG64 seed {w['seed']}",
            "l2": "inputs/outputs per step (basis 2x, coarse matrix) exceed the 126 MB L2",
            "parallelism": "patches"}


DUMP_PATCHES = 1024       # patches sampled by --dump-outputs (all of them on smaller meshes)
DUMP_SEED = 20261020
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, ctx, phi, aphi, K):
    """Write the outputs of the last timed step for a fixed, seeded sample of patches (the full arrays exceed 1 GB on
    the default workload), all float64:
      patch_ids.npy [P]             sampled patch ids, ascending
      phi.npy       [P, s, F]       basis functions; F = largest n_fine of the sample, zero past each patch's n_fine
      aphi.npy      [P, s, F]       A * basis functions, same layout
      K_ell.npy     [P * s, W]      block-ELL rows spacedim*patch + comp of the coarse matrix (layout: include/slod.h)"""
    import torch
    n, s = ctx.n_patches, phi.shape[1]
    rs = np.random.default_rng(DUMP_SEED)
    ids = np.sort(rs.choice(n, size=min(n, DUMP_PATCHES), replace=False))
    nf = np.array([ctx.patch_info(int(p))["n_fine"] for p in ids])
    width = int(nf.max())
    keep = torch.from_numpy(np.arange(width)[None, :] < nf[:, None]).to(phi.device)[:, None, :]
    sel = torch.from_numpy(ids).to(phi.device)
    rows = torch.from_numpy((ids[:, None] * s + np.arange(s)[None, :]).ravel()).to(K.device)
    arrays = {"patch_ids": ids.astype(np.float64),
              "phi": torch.where(keep, phi[sel, :, :width], 0.0).cpu().numpy(),
              "aphi": torch.where(keep, aphi[sel, :, :width], 0.0).cpu().numpy(),
              "K_ell": K[rows].cpu().numpy()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------------
def _dbg(*a):
    if os.environ.get("SLOD_BENCH_DEBUG"):
        print("[bench]", os.environ.get("RANK", "0"), *a, file=sys.stderr, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (one GPU only)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w, args.workload)
        return

    import torch
    import torch.distributed as dist
    pkg = importlib.import_module("dealii-slod_b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs needs a single-process run: phi is not gathered across ranks")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    tables = make_tables(w)
    ctx = pkg.SlodContext(dim=w["dim"], spacedim=w["s"], n_global_refinements=w["ref"], n_subdivisions=w["n"],
                          oversampling=w["ell"], stabilize=True, problem=0 if w["s"] == 1 else 1, device=local)
    for f, t in enumerate(tables):
        ctx.set_coefficient(f, w["r"], t)
    n, s, stride, ellw = ctx.n_patches, w["s"], ctx.basis_stride, ctx.ell_width
    part = importlib.import_module("dealii-slod_b200.partition")
    phi = torch.zeros((n, s, stride), dtype=torch.float64, device=dev)
    aphi = torch.zeros_like(phi)
    K = torch.zeros((n * s, ellw), dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    tk = np.zeros(8)

    # One handle per process / GPU; the two all-gathers of the phase (A*phi before the coarse rows, the K row blocks
    # after them) are NCCL calls INSIDE the library (slod_comm_init + slod_offline_distributed); torch.distributed only
    # carries the 128-byte communicator id, the barrier and the max over ranks of the measured time.
    if world > 1:
        uid = torch.tensor(list(ctx.comm_unique_id() if rank == 0 else bytes(128)), dtype=torch.uint8, device=dev)
        dist.broadcast(uid, 0)
        ctx.comm_init(rank, world, bytes(uid.cpu().numpy().tobytes()))
    p0, p1 = ctx.owned_range(rank, world)

    def step(gather_K=True):
        ctx.offline_distributed(phi.data_ptr(), aphi.data_ptr(), K.data_ptr(), gather_phi=False, gather_K=gather_K,
                                stream=stream)
        ctx.synchronize()     # the step's status check, as a caller would do it
        tk[:6] = ctx.timings()[:6]
        return tk.copy()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    _dbg("warm-up")
    for _ in range(args.warmup):
        step()
    barrier()
    _dbg("timed region")
    l0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ksum = np.zeros(8)
    with ClockSampler(local) as clk:
        e0.record()
        for _ in range(args.steps):
            ksum += step()
        e1.record()
        barrier()
    ms_total = e0.elapsed_time(e1)
    _dbg("timed done", ms_total)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ctx, phi, aphi, K)
    launches = ctx.launch_count - l0
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = n / (ms_step * 1e-3)
    kms = ksum / args.steps          # per-step kernel times of this rank (ms)

    # ---- end to end: host buffers in, host buffers out, every copy inside the timed region ----
    # N = 1: the host-buffer C ABI (what the reference's LOD::run would call).  N > 1: every rank uploads the
    # coefficient through the C ABI, computes its patch range, takes part in the A*phi all-gather, and brings its own
    # rows of phi, A*phi and K back into pinned host memory; time = max over ranks.
    e2e = None
    if not args.no_e2e:
        h2d = sum(t_.size * 8 for t_ in tables) * (2 ** (w["dim"] * max(0, w["ref"] + int(np.log2(w["n"])) - w["r"])))
        if world == 1:
            def e2e_step():
                for f, tb in enumerate(tables):
                    ctx.set_coefficient(f, w["r"], tb)
                ctx.compute_basis()
                ctx.assemble_coarse()            # enqueues; the basis read-back below overlaps the coarse kernels
                ph, _ = ctx.all_basis(reuse=True, want_aphi=False)   # the host keeps phi and K; A*phi is an intermediate
                rowptr, col, val = ctx.coarse_csr(reuse=True)
                e2e_bytes[0] = val.nbytes + ph.nbytes
                return float(val[0] + ph[0, 0, 0])
            e2e_bytes = [0]
            d2h = None
            path = "slod_set_coefficient+slod_compute_basis+slod_assemble_coarse+slod_get_all_basis(phi)+slod_get_coarse_csr"
        else:
            h_phi = torch.empty((p1 - p0, s, stride), dtype=torch.float64, pin_memory=True)
            h_K = torch.empty(((p1 - p0) * s, ellw), dtype=torch.float64, pin_memory=True)

            trace = os.environ.get("SLOD_E2E_TRACE") and rank == 0

            def e2e_step():
                tt = [time.perf_counter()]
                for f, tb in enumerate(tables):
                    ctx.set_coefficient(f, w["r"], tb)
                tt.append(time.perf_counter())
                # the library copies the rank's rows of phi / K into the pinned buffers on its own stream as soon as they
                # are final (phi while the all-gather and the coarse kernel still run); K is all-gathered on the devices
                ctx.set_host_outputs(h_phi.data_ptr(), 0, h_K.data_ptr())
                ctx.offline_distributed(phi.data_ptr(), aphi.data_ptr(), K.data_ptr(), gather_phi=False, gather_K=True,
                                        stream=stream)
                tt.append(time.perf_counter())
                ctx.synchronize()
                tt.append(time.perf_counter())
                ctx.set_host_outputs(0, 0, 0)
                torch.cuda.synchronize()
                tt.append(time.perf_counter())
                if trace:
                    print("e2e trace ms: set_coefficient %.2f  enqueue %.2f  slod_synchronize %.2f  cuda sync %.2f" %
                          tuple(1e3 * (b_ - a_) for a_, b_ in zip(tt[:-1], tt[1:])), file=sys.stderr, flush=True)
                return float(h_K[0, 0] + h_phi[0, 0, 0])
            d2h = (p1 - p0) * s * (ellw + stride) * 8 * world
            path = ("per rank: slod_set_coefficient + slod_offline_distributed (NCCL all-gather of A*phi inside the library) + "
                    "coarse rows + NCCL all-gather of K on the devices, D2H of the rank's own rows of phi and K into pinned memory "
                    "overlapped by the library (row-distributed result, as an MPI host holds it)")
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        reps = max(1, min(args.steps, 3))
        for _ in range(reps):
            e2e_step()
        barrier()
        dt = torch.tensor([(time.perf_counter() - t0) / reps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dt = float(dt.item())
        if d2h is None:
            d2h = e2e_bytes[0]   # CSR values + phi + A*phi (rowptr / col are integer geometry cached on the host)
        e2e = {"value": n / dt, "unit": "patches/s", "h2d_bytes_per_step": int(h2d) * world,
               "d2h_bytes_per_step": int(d2h), "ms_per_step": dt * 1e3, "path": path}

    # Online phase on the handle's own basis and coarse matrix (SURVEY 8f row 1): informational, outside the metric.
    # f = 1 per component (closed form of the Gauss sums: h^dim at interior nodes, 0 on the boundary).
    online = None
    if e2e is not None and world == 1:
        G = (2 ** w["ref"]) * w["n"] + 1
        w1 = np.full(G, 1.0 / (G - 1))
        w1[0] = w1[-1] = 0.0
        f = w1
        for _ in range(w["dim"] - 1):
            f = np.multiply.outer(w1, f)
        f = np.repeat(f.ravel(), s)
        ctx.prolongate(ctx.coarse_solve(ctx.coarse_rhs(f), max_steps=5, tolerance=0.0, reduction=1e9)[0])   # first-launch costs (one CG step)
        t0 = time.perf_counter()
        b = ctx.coarse_rhs(f)
        t1 = time.perf_counter()
        u, cg_steps, cg_res = ctx.coarse_solve(b, max_steps=20000, tolerance=0.0, reduction=1e-10)
        t2 = time.perf_counter()
        uh = ctx.prolongate(u)
        t3 = time.perf_counter()
        online = {"coarse_rhs_ms": (t1 - t0) * 1e3, "coarse_cg_ms": (t2 - t1) * 1e3, "cg_steps": int(cg_steps),
                  "cg_reduction": 1e-10, "cg_residual": float(cg_res), "prolongate_ms": (t3 - t2) * 1e3,
                  "u_fine_l2": float(np.linalg.norm(uh)),
                  "note": "host-buffer C ABI calls (copies included), forcing f = 1, diag(K)-preconditioned CG"}

    # ---- N > 1: the distributed result against a single-GPU recomputation on rank 0 (outside the timed region) ----
    multi_gpu_check = None
    _dbg("e2e done")
    if os.environ.get("SLOD_BENCH_DEBUG"):
        import faulthandler
        faulthandler.dump_traceback_later(45, exit=True)
    if world > 1:
        ctx.offline_distributed(phi.data_ptr(), aphi.data_ptr(), K.data_ptr(), gather_phi=True, gather_K=True, stream=stream)
        ctx.synchronize()
        torch.cuda.synchronize()
        _dbg("check: distributed step done")
        if rank == 0:
            # patches of a sub-range that straddles the first partition boundary, recomputed by this rank alone into
            # fresh buffers; the coarse rows of the range need A*phi of their neighbours: take it from the gathered array
            half = max(1, min(64, (p1 - p0) // 2))
            q0, q1 = p1 - half, min(n, p1 + half)
            phi2 = torch.zeros_like(phi)
            aphi2 = torch.zeros_like(aphi)
            _dbg("check: buffers allocated")
            ctx.compute_basis_device(q0, q1, phi2.data_ptr(), aphi2.data_ptr(), stream)
            ctx.synchronize()
            _dbg("check: basis recomputed")
            same_phi = bool(torch.equal(phi2[q0:q1], phi[q0:q1]))
            same_aphi = bool(torch.equal(aphi2[q0:q1], aphi[q0:q1]))
            K2 = torch.zeros_like(K)
            ctx.assemble_coarse_device(q0, q1, phi.data_ptr(), aphi.data_ptr(), K2.data_ptr(), stream)
            ctx.synchronize()
            same_K = bool(torch.equal(K2[q0 * s:q1 * s], K[q0 * s:q1 * s]))
            multi_gpu_check = {"range": [int(q0), int(q1)], "phi_bit_equal": same_phi, "aphi_bit_equal": same_aphi,
                               "K_rows_bit_equal": same_K,
                               "note": "rank 0 recomputes patches on both sides of the first partition boundary on its own "
                                       "and compares with the all-gathered result"}
            if not (same_phi and same_aphi and same_K):
                raise SystemExit(f"multi-GPU result differs from the single-GPU recomputation: {multi_gpu_check}")
            del phi2, aphi2, K2
        # The other ranks wait on the HOST (the rendezvous store), not in an NCCL barrier: a collective kernel spinning
        # on their GPUs while rank 0 allocates memory (cudaMalloc synchronises with peer-mapped devices) deadlocks.
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            store.set("slod_check_done", "1")
        else:
            store.wait(["slod_check_done"])
        barrier()

    _dbg("check done")
    if rank == 0:
        fm = flop_model(w)
        names = ["patch_solve", "patch_dense", "patch_select", "patch_finish"]
        share = (p1 - p0) / n
        kern = {}
        for i, nm in enumerate(names):
            if kms[i] > 0:
                kern[nm] = {"ms": float(kms[i]), "tflops": fm[nm] * share / (kms[i] * 1e-3) / 1e12}
        kern["coarse"] = {"ms": float(kms[4])}
        if kms[5] > 0:
            kern["patch_solve"]["factor_ms"] = float(kms[5])
            kern["patch_solve"]["trisolve_ms"] = float(kms[0] - kms[5])
        dom = max(names, key=lambda nm: kms[names.index(nm)])
        achieved = kern[dom]["tflops"]
        kname = {"patch_solve": "k_patch_factor + k_patch_trisolve" if kms[5] > 0 else "k_patch_solve_mma", "patch_dense": "k_patch_flux + k_patch_dense_mma",
                 "patch_select": "k_select_fast + k_eig_tridiag/ql/finish", "patch_finish": "k_patch_finish"}[dom]
        traffic = None
        tfile = os.path.join(ROOT, "profiles", "dram_traffic.json")   # per-launch DRAM bytes from the committed ncu capture
        if os.path.exists(tfile) and args.workload == DEFAULT_WORKLOAD and world == 1:
            tr = json.load(open(tfile))
            traffic = tr.get(kname, tr.get(kname.split(" ")[0]))
        # FP64 peak of THIS device, measured now (same process, after the timed region) with the library's probe kernels
        peak, peak_src = FP64_PEAK_FALLBACK, "fallback constant (probe failed)"
        try:
            with ClockSampler(local) as pclk:
                dfma, dmma = ctx.measure_fp64_peak()
            peak = max(dfma, dmma)
            peak_src = (f"slod_measure_fp64_peak in this run: DFMA {dfma:.2f}, mma.sync m8n8k4 f64 {dmma:.2f} TFLOP/s "
                        f"at {pclk.summary()['sm_mhz']} MHz (MEASURED_PEAKS.json has no fp64 entry)")
        except Exception as exc:   # noqa: BLE001
            peak_src += f": {exc}"
        roofline = {"bound": "tensor", "pipe": "fp64 (DFMA/DMMA share one pipe on B200)", "kernel": kname,
                    "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                    "traffic": traffic, "peak_source": peak_src,
                    "flop_model": "banded Cholesky Ni*bw^2 + 4*Ni*bw*Ncd per patch (SURVEY 8d), summed over actual patch shapes",
                    "kernels": kern}
        for nm in kern:
            if "tflops" in kern[nm]:
                kern[nm]["frac"] = kern[nm]["tflops"] / peak
        cpu = None
        parity = None
        if not args.no_cpu_baseline and world == 1:
            rate, dt, cpu_h, ids = cpu_port_step(w, tables, 0)
            cpu = {"value": rate, "unit": "patches/s", "cores": cpu_h.threads, "kind": "port", "language": "c++",
                   "seconds": dt, "sample": cpu_sample_text(w, ids.size, cpu_h.threads)}
            # the same patches from the GPU run, compared outside the timed region
            step()
            gpu_csr = None
            if e2e is not None:
                ctx.compute_basis()
                ctx.assemble_coarse()
                gpu_csr = ctx.coarse_csr(reuse=True)
            parity = parity_against_cpu(w, cpu_h, ids, phi, aphi, gpu_csr, lambda pid, d: ctx.diagnostics(pid, d))
            cpu_h.close()
        line = {"metric": "slod_basis_patches_per_s", "value": value, "unit": "patches/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config_of(w, args.workload), "clocks": clk.summary(), "e2e": e2e,
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "parity_max": parity,
                "multi_gpu_check": multi_gpu_check, "offline_wall_ms": ms_step, "online": online}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
