"""Double against Single "Subdomain Inverse Precision" on the bench default problem, one GPU, in one process:

    python tools/a11_precision_timing.py [--nx 128] [--reps 30] [--rounds 3] [--out FILE.json]

Workload: the problem of bench.py (Stokes-C 128^3, skew partitioner, sx = 8, cx = 4, 2 levels; b = A x_ex with x_ex
uniform(-1, 1) seed 42, GMRES from x0 uniform(-1, 1) seed 43 to 1e-8).  Two handles on the same matrix, one per
precision, both resident while the timed rounds alternate their order.  Per handle and round:
  * apply_ms: ApplyInverse on device vectors (hymls_b200_time_apply, CUDA events over `reps` calls);
  * a11_full_pass_ms / a11_full_pass_gbs: the level-0 full-pass GEMV kernel (CUDA events around every launch) and
    bytes_a11_full_pass over it;
  * host_apply_per_s: ApplyInverse calls per second with pinned host buffers (host clock, synchronised).
Then ||x_single - x_double|| / ||x_double|| of one ApplyInverse, and GMRES once per precision on a fresh handle, one
at a time (iterations, seconds, explicit residual, the same difference of the solutions).  The card's name and power limit are read in the same run.
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import hymls_b200 as hb  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def host_rate(P, b, reps):
    import torch
    n = len(b)
    hin = torch.from_numpy(b).pin_memory()
    hout = torch.empty(n, dtype=torch.float64).pin_memory()
    lib, h = P._lib, P._h
    for _ in range(2):
        hb.api._check(lib, lib.hymls_b200_apply_inverse(h, hin.data_ptr(), n, hout.data_ptr(), n, 1, hb.api.HOST))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        lib.hymls_b200_apply_inverse(h, hin.data_ptr(), n, hout.data_ptr(), n, 1, hb.api.HOST)
    torch.cuda.synchronize()
    return reps / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=128)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    torch.cuda.set_device(0)
    params = bench.make_params(args.nx, 8, 2, 4)
    A, tv, _, b, x0 = bench.problem(args.nx)
    handles, setup = {}, {}
    for prec in ("Double", "Single"):
        p = copy.deepcopy(params)
        p["Preconditioner"]["Subdomain Inverse Precision"] = prec
        P = hb.Preconditioner(A, p, tv)
        P.Initialize()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        P.Compute()
        torch.cuda.synchronize()
        st = P.Stats()
        setup[prec] = {"compute_s": time.perf_counter() - t0, "a11_entry_bytes": st["a11_entry_bytes"],
                       "bytes_a11_full_pass": st["bytes_a11_full_pass"], "bytes_a11_level0": st["bytes_a11_level0"],
                       "bytes_apply": st["bytes_apply"], "device_bytes": st["device_bytes"]}
        handles[prec] = P
    res = {prec: {"apply_ms": [], "a11_full_pass_ms": [], "a11_full_pass_gbs": [], "host_apply_per_s": []}
           for prec in handles}
    for r in range(args.rounds):
        for prec in (("Double", "Single") if r % 2 == 0 else ("Single", "Double")):
            P = handles[prec]
            ms_apply, ms_a11 = P.TimeApply(args.reps)
            res[prec]["apply_ms"].append(ms_apply)
            res[prec]["a11_full_pass_ms"].append(ms_a11)
            res[prec]["a11_full_pass_gbs"].append(setup[prec]["bytes_a11_full_pass"] / (ms_a11 * 1e-3) / 1e9)
            res[prec]["host_apply_per_s"].append(host_rate(P, b, args.reps))
    x = {prec: handles[prec].ApplyInverse(b) for prec in handles}
    # GMRES(600) holds 600 basis vectors (40 GB at 128^3) per handle: one handle at a time
    handles.clear()
    del P
    gm, xs = {}, {}
    for prec in ("Double", "Single"):
        p = copy.deepcopy(params)
        p["Preconditioner"]["Subdomain Inverse Precision"] = prec
        P = hb.Preconditioner(A, p, tv)
        P.Initialize()
        P.Compute()
        S = hb.Solver(P)
        xs[prec] = S.ApplyInverse(b, x0.copy())
        gm[prec] = {"iterations": S.num_iter, "converged": bool(S.info["converged"]),
                    "solve_s": S.info["solve_seconds"], "explicit_rel_residual": S.info["explicit_rel_residual"]}
        del S, P
    out = {"card": card(), "n": int(A.shape[0]), "nx": args.nx, "sx": 8, "cx": 4, "levels": 2,
           "partitioner": bench.PARTITIONER, "reps": args.reps, "rounds": args.rounds, "setup": setup,
           "timing": res,
           "median": {prec: {k: float(np.median(v)) for k, v in res[prec].items()} for prec in res},
           "gmres": gm,
           "apply_rel_diff_single_vs_double": float(np.linalg.norm(x["Single"] - x["Double"]) /
                                                    np.linalg.norm(x["Double"])),
           "gmres_solution_rel_diff": float(np.linalg.norm(xs["Single"] - xs["Double"]) /
                                            np.linalg.norm(xs["Double"]))}
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
