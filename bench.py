#!/usr/bin/env python
"""Headline benchmark: HYMLS preconditioner hot path on a synthetic 3D lid-driven-cavity (Stokes-C)
Jacobian, BASELINE.json's metric "ApplyInverse/s + HBM GB/s; GMRES solve time".

    python bench.py --gpus N --steps K --warmup W            # this implementation (CUDA, sm_100a)
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the reference's algorithm restated in
                                                             # C++/OpenMP (oracle/cpp), all host threads

A "step" is one Preconditioner::ApplyInverse on one right-hand side.  `value` is ApplyInverse/s with the vectors
resident in HBM; `e2e` is the same call through the C ABI with pinned HOST buffers (H2D of b and D2H of x inside the
timed region).  One JSON line is printed by rank 0.  With --dump-outputs DIR, rank 0 also writes the vector the last
timed ApplyInverse returned and the GMRES solution as DIR/apply_inverse_x.npy and DIR/gmres_x.npy (float64; a fixed
sample of rows, listed in DIR/rows.npy, when they would exceed 64 MB).  The inputs depend only on the arguments, so two
builds, or the two arms, can be compared file by file.

Multi-GPU (torchrun, one rank per GPU): ONE problem ("scaling": "strong"), its subdomains distributed over the ranks
by the reference's subdomain -> rank map (CreatePIDMap); vectors are distributed by row owner; only separator values
on the interfaces between ranks (grouped ncclSend/ncclRecv), the V-sums and the Krylov dot products cross NVLink.
Timing is the max over ranks.  With N > 1 the line also carries `mgpu_check`: sharded vs single-GPU ApplyInverse /
GMRES on a small problem run inside the same job.

The CPU arm runs the SAME parameter list (levels, cx, partitioner) on the same workload when the host can hold it
(--cpu-nx, default: the workload's nx for --gpus 1 with >= 16 cores and >= 96 GB of free RAM, else 64) for K real ApplyInverse
calls and the GMRES solve; on a smaller grid the rate is scaled by the subdomain ratio and flagged.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DMMA_PEAK_TFLOPS = 37.1  # measured FP64 tensor (mma.sync.m8n8k4.f64) peak, profiles/r01_dmma_microbench.txt


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="hymls_b200", choices=["hymls_b200", "reference"])
    ap.add_argument("--nx", type=int, default=int(os.environ.get("HYMLS_BENCH_NX", 128)))
    ap.add_argument("--sx", type=int, default=int(os.environ.get("HYMLS_BENCH_SX", 8)))
    ap.add_argument("--levels", type=int, default=2)
    ap.add_argument("--cx", type=int, default=4, help="coarsening factor between levels")
    ap.add_argument("--partitioner", default="Skew Cartesian", choices=["Skew Cartesian", "Cartesian"],
                    help="'Skew Cartesian' is what the reference uses for 3D Stokes; 'Cartesian' needs the "
                         "documented tube-pressure extension (DESIGN.md, Deviations)")
    ap.add_argument("--no-solve", action="store_true", help="skip the GMRES solve")
    ap.add_argument("--no-check", action="store_true", help="skip the sharded-vs-single check of multi-GPU runs")
    ap.add_argument("--cpu-nx", type=int, default=0, help="grid of the CPU arm (0: automatic)")
    ap.add_argument("--cpu-sample-nx", type=int, default=64,
                    help="grid of the cpu_baseline leg of the GPU arm (64^3: 1296 of the 9248 subdomains, ~15 s of CPU "
                         "work; its factors no longer fit the caches, like the full size)")
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the ApplyInverse result of the last timed step (and the GMRES "
                         "solution) as DIR/<name>.npy in float64, for comparing two builds on the same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT_BYTES):
    """Writes each vector of `arrays` (name -> 1-D array, all of one length) as out_dir/<name>.npy in float64.  When
    they would exceed `limit` bytes in all, every file holds the same rows: a fixed sample (numpy seed 0, ascending),
    whose indices go to out_dir/rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(next(iter(arrays.values())))
    rows = None
    if 8 * n * len(arrays) > limit - 4096:                  # (4096: room for the .npy headers)
        k = (limit - 4096) // (8 * (len(arrays) + 1))
        rows = np.sort(np.random.default_rng(0).choice(n, k, replace=False))
        arrays = dict(rows=rows, **{name: np.asarray(v)[rows] for name, v in arrays.items()})
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(v, dtype=np.float64))


PARTITIONER = "Skew Cartesian"


def make_params(nx, sx, levels, cx):
    prec = {"Partitioner": PARTITIONER, "Separator Length": sx, "Number of Levels": levels,
            "Coarsening Factor": cx}
    if PARTITIONER == "Cartesian":
        prec["Eliminate Tube Pressures With Velocities"] = True
    return {
        "Problem": {"Equations": "Stokes-C", "Dimension": 3, "nx": nx, "ny": nx, "nz": nx},
        "Preconditioner": prec,
        # the initial vector is passed in explicitly (uniform(-1,1), numpy seed 43) so that both arms start from
        # the same x0 and their residual histories can be compared entry by entry
        "Solver": {"Krylov Method": "GMRES", "Initial Vector": "Previous", "Left or Right Preconditioning": "Right",
                   "Iterative Solver": {"Maximum Iterations": 600, "Num Blocks": 600, "Maximum Restarts": 0,
                                        "Convergence Tolerance": 1e-8,
                                        "Implicit Residual Scaling": "Norm of Initial Residual"}},
    }


def num_subdomains(nx, sx):
    npx = nx // sx
    return npx ** 3 if PARTITIONER == "Cartesian" else (2 * npx * npx + 2 * npx) * (npx + 1)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            try:
                sm.append(float(f[0]))
                smax.append(float(f[1]))
            except Exception:
                continue
            for name, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def ncu_traffic(alg_bytes):
    """dram__bytes_read.sum + dram__bytes_write.sum of one level-0 k_batched_gemv launch from the committed
    `ncu --set full` capture, if it was taken on this workload."""
    for name in ("r02_ncu_gemv_traffic.json", "r01_ncu_gemv_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                t = json.load(f)
            if abs(t["algorithmic_bytes_per_launch"] - alg_bytes) <= 1e-6 * alg_bytes:
                return t["dram_bytes_per_launch"]
        except Exception:
            pass
    return None


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md, 6.65 TB/s)"


def problem(nx):
    """the synthetic Jacobian, the exact solution / right-hand side (seed 42) and the initial vector (seed 43)"""
    import hymls_b200.galeri as galeri
    A = -galeri.create_matrix("Stokes-C", 3, nx)
    tv = galeri.create_testvector(A)
    n = A.shape[0]
    xex = np.random.default_rng(42).uniform(-1, 1, n)
    x0 = np.random.default_rng(43).uniform(-1, 1, n)
    return A, tv, xex, A @ xex, x0


def host_cores():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def mem_available_gb():
    try:
        with open("/proc/meminfo") as f:
            for ln in f:
                if ln.startswith("MemAvailable"):
                    return float(ln.split()[1]) / 1e6
    except Exception:
        pass
    return 0.0


def cpu_oracle_run(nx, sx, levels, cx, steps, warmup, threads, solve):
    """The reference's CPU path restated in C++/OpenMP (oracle/cpp/hymls_oracle.cpp) on the grid `nx`: Compute,
    `steps` ApplyInverse calls, optionally the GMRES solve.  The index maps come from the library's HOST
    partitioner (no GPU; bit-exact with oracle/partitioner.py, tests/test_host_maps.py).  Besides the figures, the
    result holds the vectors computed: "x" (last ApplyInverse) and "gmres_x" (GMRES solution, if solved)."""
    import hymls_b200 as hb
    from oracle import cpp_oracle as oc
    from oracle.params import ParameterList

    def to_pl(d):
        pl = ParameterList()
        for k, v in d.items():
            pl[k] = to_pl(v) if isinstance(v, dict) else v
        return pl

    t0 = time.time()
    A, tv, xex, b, x0 = problem(nx)
    p = make_params(nx, sx, levels, cx)
    P = hb.Preconditioner(A, p, tv, pattern_only=True)
    P.Initialize()
    maps = oc.maps_from_library(P)
    del P
    t_setup = time.time() - t0
    O = oc.Preconditioner(A, to_pl(p), tv, maps, threads=threads)
    del maps
    t0 = time.time()
    O.compute()
    t_compute = time.time() - t0
    for _ in range(max(1, min(warmup, 3))):
        x = O.apply_inverse(b)
    t0 = time.time()
    for _ in range(steps):
        x = O.apply_inverse(b)
    t_apply = (time.time() - t0) / steps
    st = O.stats()
    out = {"nx": nx, "n": int(A.shape[0]), "subdomains": num_subdomains(nx, sx), "threads": st["threads"],
           "setup_s": t_setup, "compute_s": t_compute, "factor_a11_s": st["factor_a11_s"], "schur_s": st["schur_s"],
           "apply_s": t_apply, "nnz_factors": st["nnz_factors"], "apply_checksum": float(np.linalg.norm(x)), "x": x}
    if solve:
        it = p["Solver"]["Iterative Solver"]
        xs, its, conv, hist, sec = O.solve(b, x0=x0, method="GMRES", tol=it["Convergence Tolerance"],
                                           max_iters=it["Maximum Iterations"], num_blocks=it["Num Blocks"],
                                           max_restarts=it["Maximum Restarts"])
        out["gmres"] = {"iterations": its, "converged": bool(conv), "solve_s": sec,
                        "explicit_rel_residual": float(np.linalg.norm(A @ xs - b) / np.linalg.norm(b)),
                        "rel_error": float(np.linalg.norm(xs - xex) / np.linalg.norm(b)),
                        "history_first15": [float(v) for v in hist[:15]], "tol": it["Convergence Tolerance"]}
        out["gmres_x"] = xs
    return out


def reference_arm(args, workload):
    cores = host_cores()
    threads = args.cpu_threads or cores
    nx_cpu = args.cpu_nx
    if nx_cpu <= 0:
        # the full workload takes ~4 minutes on 16 cores (Compute ~45 s, GMRES ~3 min): run it for the N=1 line; the
        # lines of a scaling run (N > 1, same CPU quantity every time) use the 64^3 grid scaled by the subdomain ratio
        # (fewer than 16 cores would push the full-size run beyond ~5 minutes)
        full = cores >= 16 and mem_available_gb() >= 96.0 and args.gpus == 1
        nx_cpu = args.nx if full else min(args.nx, 64)
    r = cpu_oracle_run(nx_cpu, args.sx, args.levels, args.cx, args.steps, args.warmup, threads, not args.no_solve)
    same = nx_cpu == args.nx
    scale = r["subdomains"] / float(num_subdomains(args.nx, args.sx))   # time is linear in the subdomain count
    v = scale / r["apply_s"]
    sample = ("C++/OpenMP restatement of the reference's CPU path (oracle/cpp: sparse LU per subdomain in the "
              "reference's F-matrix ordering, same parameter list), %d threads, %d^3 grid = %d of %d subdomains%s: Compute %.1f s, %d timed ApplyInverse "
              "calls at %.1f ms" % (r["threads"], nx_cpu, r["subdomains"], num_subdomains(args.nx, args.sx),
                                    "" if same else " (rate scaled by the subdomain ratio)", r["compute_s"],
                                    args.steps, r["apply_s"] * 1e3))
    out = {"impl": "reference", "metric": "apply_inverse_per_s", "value": v, "unit": "1/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / v, "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": workload, "parallelism": "cpu: 1 process x %d OpenMP threads" % r["threads"],
                      "same_config": same, "extrapolated": not same, "cpu_nx": nx_cpu,
                      "t_compute_s": r["compute_s"], "gmres": r.get("gmres")},
           "cpu_baseline": {"value": v, "unit": "1/s", "cores": r["threads"], "kind": "port", "sample": sample,
                            "apply_ms_measured": r["apply_s"] * 1e3, "compute_s": r["compute_s"],
                            "factor_a11_s": r["factor_a11_s"], "schur_assembly_s": r["schur_s"],
                            "nnz_subdomain_factors": r["nnz_factors"], "gmres": r.get("gmres")},
           "e2e": {"value": v, "unit": "1/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gmres": r.get("gmres")}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: v for k, v in (("apply_inverse_x", r["x"]), ("gmres_x", r.get("gmres_x")))
                                         if v is not None})
    print(json.dumps(out))


def main():
    global PARTITIONER
    args = parse()
    PARTITIONER = args.partitioner
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    nx, sx = args.nx, args.sx
    cx = args.cx
    workload = ("synthetic 3D lid-driven cavity (Stokes-C, GaleriExt::Stokes3D a=nx^2 b=1) %d^3, dof 4, %s partitioner, "
                "sx=%d, %d levels, cx=%d" % (nx, PARTITIONER, sx, args.levels, cx))

    if args.impl == "reference":
        if rank == 0:   # the other ranks of a torchrun launch exit without work
            reference_arm(args, workload)
        return

    import torch
    import hymls_b200 as hb

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    t0 = time.time()
    A, tv, xex, bh, x0h = problem(nx)
    t_gen = time.time() - t0
    n = A.shape[0]
    P = hb.Preconditioner(A, make_params(nx, sx, args.levels, cx), tv)
    if world > 1:
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(hb.Preconditioner.CommUniqueId()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        P.CommInit(bytes(idt.cpu().numpy().tobytes()), rank, world)
    t0 = time.time()
    P.Initialize()
    t_init = time.time() - t0
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()  # ranks leave the (host-side) Initialize at different times: do not bill that to Compute
    t0 = time.time()
    P.Compute()
    torch.cuda.synchronize()
    t_compute = time.time() - t0
    # a Newton solver recomputes the preconditioner on every step with the same pattern: the second Compute reuses the
    # scratch the first one allocated
    if dist is not None:
        dist.barrier()
    t0 = time.time()
    P.Compute()
    torch.cuda.synchronize()
    t_recompute = time.time() - t0
    st = P.Stats()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing (value): vectors distributed by row owner, resident in HBM ----
    rows = P.OwnedRows()
    b_own = torch.from_numpy(bh[rows]).cuda()
    for _ in range(max(args.warmup, 3)):
        x_own = P.ApplyInverseDist(b_own)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = P.Stats()["kernel_launches"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    lib, h = P._lib, P._h
    x_own = torch.empty_like(b_own)
    e0.record()
    for _ in range(args.steps):
        lib.hymls_b200_apply_inverse_dist(h, b_own.data_ptr(), x_own.data_ptr(), 1)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = P.Stats()["kernel_launches"] - l0
    # ---- end-to-end through the C ABI with pinned host buffers: every rank passes / receives the rows it owns
    #      of the (distributed) vectors, like the reference's Epetra_MultiVector on an MPI rank ----
    hb_in = torch.empty(len(rows), dtype=torch.float64).pin_memory()
    hb_out = torch.empty(len(rows), dtype=torch.float64).pin_memory()
    hb_in.copy_(torch.from_numpy(bh[rows]))
    bin_np, bout_np = hb_in.numpy(), hb_out.numpy()
    for _ in range(2):
        rc = lib.hymls_b200_apply_inverse_dist(h, bin_np.ctypes.data, bout_np.ctypes.data, 0)
        if rc != 0:
            raise RuntimeError("apply_inverse_dist (host buffers): " + lib.hymls_b200_last_error().decode())
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        lib.hymls_b200_apply_inverse_dist(h, bin_np.ctypes.data, bout_np.ctypes.data, 0)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    e2e_ok = bool(np.array_equal(bout_np, x_own.cpu().numpy()))
    clocks = sampler.stop()
    st_e2e = P.Stats()   # (host_pipeline_state as the timed loop left it)
    # the same loop with the copy / compute overlap of the host-buffer path switched off (one GPU; the switch is read
    # at every call): the serial-copies figure next to the default one
    e2e_serial_ms = None
    if world == 1:
        old_env = os.environ.get("HYMLS_B200_HOST_PIPELINE")
        os.environ["HYMLS_B200_HOST_PIPELINE"] = "0"
        try:
            for _ in range(2):
                lib.hymls_b200_apply_inverse_dist(h, bin_np.ctypes.data, bout_np.ctypes.data, 0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                lib.hymls_b200_apply_inverse_dist(h, bin_np.ctypes.data, bout_np.ctypes.data, 0)
            torch.cuda.synchronize()
            e2e_serial_ms = (time.perf_counter() - t0) * 1e3
        finally:
            if old_env is None:
                del os.environ["HYMLS_B200_HOST_PIPELINE"]
            else:
                os.environ["HYMLS_B200_HOST_PIPELINE"] = old_env
    # ---- dominant kernel (batched A11^-1 apply, level 0) via CUDA events inside the library ----
    ms_apply_lib, ms_a11 = P.TimeApply(max(5, min(args.steps, 20)))
    st2 = P.Stats()
    # ---- GMRES solve (the other half of the metric) ----
    gm = None
    if not args.no_solve:
        S = hb.Solver(P)
        bd, xd = torch.from_numpy(bh).cuda(), torch.from_numpy(x0h).cuda()
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        xs = S.ApplyInverse(bd, x=xd)
        torch.cuda.synchronize()
        solve_wall = time.perf_counter() - t0   # first call: includes the one-off allocation of the Krylov basis
        err = float(np.linalg.norm(xs.cpu().numpy() - xex) / np.linalg.norm(bh))
        gm = {"iterations": S.num_iter, "converged": bool(S.info["converged"]),
              "solve_s": S.info["solve_seconds"], "solve_wall_first_call_s": solve_wall,
              "explicit_rel_residual": S.info["explicit_rel_residual"],
              "rel_error": err, "tol": 1e-8, "restart": "none (Num Blocks 600)",
              "history_first15": [float(v) for v in S.history[:15]]}
    # ---- multi-GPU: sharded vs single-GPU results on a small problem, inside the same job ----
    check = None
    if world > 1 and not args.no_check:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        from mgpu_check import run_check
        try:
            check = run_check(32, 8, 2, 2, PARTITIONER, rank, world)
        except Exception as e:   # the check must not cost the bench line
            check = {"error": repr(e)}

    tm = torch.tensor([ms, e2e_ms, ms_a11, t_compute, gm["solve_s"] if gm else 0.0], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms, e2e_ms, ms_a11, t_compute, solve_s = [float(v) for v in tm.cpu()]
    if gm:
        gm["solve_s"] = solve_s
    if args.dump_outputs:
        # the result of the last timed step, assembled from the rows each rank owns
        x_full = torch.zeros(n, dtype=torch.float64, device="cuda")
        x_full[torch.from_numpy(rows).cuda()] = x_own
        if dist is not None:
            dist.all_reduce(x_full)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"apply_inverse_x": x_full.cpu().numpy(),
                                             **({"gmres_x": xs.cpu().numpy()} if gm else {})})
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak_gbs()
    # one pass over the explicit A11 inverses this rank owns (SURVEY 8(d): 8 n_sd^2 bytes per subdomain solve)
    alg_bytes = st["bytes_a11_full_pass"]
    split = bool(st.get("a11_split", 0))
    # (split second solve: the timed kernel is the leading-columns pass, 8 sum n nb bytes)
    lead_bytes = alg_bytes if split else st["bytes_a11_level0"] - alg_bytes
    full_bytes = st["bytes_a11_level0"] - lead_bytes
    achieved = alg_bytes / (ms_a11 * 1e-3) / 1e9 if ms_a11 > 0 else 0.0
    value = args.steps / (ms * 1e-3)
    compute_tflops = st["flops_compute"] / t_compute / 1e12
    out = {
        "metric": "apply_inverse_per_s", "value": value, "unit": "1/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload, "n": n, "nnz": int(A.nnz), "subdomains": int(st["num_subdomains"]),
                   "parallelism": ("subdomains distributed over %d ranks (CreatePIDMap), vectors by row owner; separator "
                                   "halo by grouped ncclSend/ncclRecv, V-sum and dot-product all-reduces" % world)
                   if world > 1 else "single GPU",
                   "l2": ("inputs larger than L2 (A11 inverses %.2f GB per rank; per step: leading rows %.2f GB, then the "
                          "remaining rows %.2f GB on a low-priority stream beside the separator phase, then the leading "
                          "columns %.2f GB)" % (full_bytes / 1e9, lead_bytes / 1e9, (full_bytes - lead_bytes) / 1e9,
                                                lead_bytes / 1e9)) if split else
                         ("inputs larger than L2 (A11 inverses %.2f GB per rank: one full pass + a %.2f GB pass over "
                          "their leading rows per step)" % (full_bytes / 1e9, lead_bytes / 1e9)),
                   "sum_nsd_sq": st["sum_nsd_sq"], "sum_nsd_nb": st["sum_nsd_nb"],
                   "bytes_apply_algorithmic": st["bytes_apply"],
                   "apply_gbs_all_kernels": st["bytes_apply"] / (ms / args.steps * 1e-3) / 1e9,
                   "apply_frac_of_peak_all_gpus": st["bytes_apply"] / (ms / args.steps * 1e-3) / 1e9 / (peak * world),
                   "t_generate_s": t_gen, "t_initialize_s": t_init, "t_compute_s": t_compute, "t_recompute_s": t_recompute,
                   "compute_tflops": compute_tflops, "gmres": gm, "mgpu_check": check},
        "e2e": {"value": args.steps / (e2e_ms * 1e-3), "unit": "1/s", "h2d_bytes_per_step": 8 * n,
                "d2h_bytes_per_step": 8 * n, "per_rank_bytes_each_way": 8 * len(rows),
                "matches_device_result": e2e_ok,
                # one GPU: the copies are overlapped with the two passes over the level-0 inverses in `chunks` pieces
                # (state 1 = the first such call reproduced the serial path bit for bit; DESIGN.md section 3)
                "host_pipeline": {"chunks": int(st_e2e.get("host_pipeline_chunks", 0)),
                                  "state": int(st_e2e.get("host_pipeline_state", 0)),
                                  "value_with_serial_copies": (args.steps / (e2e_serial_ms * 1e-3))
                                  if e2e_serial_ms else None},
                "call": "hymls_b200_apply_inverse_dist (pinned host rows this rank owns in / out)"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": ("k_batched_gemv (A11^-1 apply, level 0, per rank: the leading-columns pass "
                                                "of the split second subdomain solve)" if split else
                                                "k_batched_gemv (A11^-1 apply, level 0, per rank: the full pass "
                                                "of the second subdomain solve)"), "achieved": achieved,
                     "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic(alg_bytes),
                     "bytes_per_launch": alg_bytes, "ms_per_launch": ms_a11, "peak_source": peak_src,
                     "leading_rows_pass": {"bytes_per_launch": lead_bytes,
                                           "ms_per_launch": st2["ms_a11_lead"],
                                           "achieved": (lead_bytes / (st2["ms_a11_lead"] * 1e-3) / 1e9)
                                           if st2["ms_a11_lead"] > 0 else 0.0},
                     "compute": {"bound": "tensor", "what": "Compute(): batched FP64 inversions + Newton-Schulz GEMMs + "
                                 "Schur assembly, all levels (algorithmic flops / wall time)", "achieved": compute_tflops,
                                 "peak": DMMA_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": compute_tflops / DMMA_PEAK_TFLOPS,
                                 "peak_source": "measured DMMA m8n8k4 microbenchmark (profiles/r01_dmma_microbench.txt)"}},
        "gmres": gm,
        "mgpu_check": check,
    }
    # CPU baseline on a bounded sample of the same workload (rank 0, N=1 only): the C++/OpenMP restatement with the
    # same parameter list on a smaller grid; work is linear in the number of subdomains
    if world == 1:
        snx = min(nx, max(args.cpu_sample_nx, 4 * sx))
        r = cpu_oracle_run(snx, sx, args.levels, cx, 10, 1, args.cpu_threads or host_cores(), False)
        scale = r["subdomains"] / float(num_subdomains(nx, sx))
        out["cpu_baseline"] = {
            "value": scale / r["apply_s"], "unit": "1/s", "cores": r["threads"], "kind": "port",
            "sample": "C++/OpenMP restatement (oracle/cpp, sparse LU per subdomain in the reference's F-matrix ordering, "
                      "same parameter list) on a %d^3 grid "
                      "= %d of %d subdomains, %d threads; 10 ApplyInverse calls at %.2f ms, rate scaled by the "
                      "subdomain ratio; `bench.py --impl reference` runs the full-size CPU arm"
                      % (snx, r["subdomains"], num_subdomains(nx, sx), r["threads"], r["apply_s"] * 1e3),
            "sample_apply_ms": r["apply_s"] * 1e3, "sample_compute_s": r["compute_s"]}
    print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
