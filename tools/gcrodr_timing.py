"""GCRO-DR ("Krylov Method" = "GCRODR") against GMRES(600) on the bench problem, one GPU, in one process:

    python tools/gcrodr_timing.py [--nx 128] [--reps 10] [--out profiles/r08_gcrodr_1gpu.json] [--md profiles/r08_gcrodr.md]

writes the JSON line and the tables of the markdown file (both paths are the defaults shown).  A "## Findings" section
of an existing markdown file is written by hand; it is kept below the regenerated tables.

Problem and inputs are the bench's (Stokes-C 128^3, skew partitioner, sx = 8, cx = 4, 2 levels; b = A x_ex, x0
uniform(-1, 1) seed 43, tolerance 1e-8 in the "Norm of Initial Residual" scaling, Right preconditioning).

  * GMRES(600), Maximum Restarts 0: the bench solve, the baseline line.
  * GCRODR(m, k) for (100, 20), (200, 30), (300, 40), Maximum Restarts 50: iterations, converged, solve_seconds, the
    explicit residual, krylov_basis_bytes and the recycled columns.
  * Restart-phase kernels at the bench's n: blockDot of m + 1 basis vectors against k + 1 vectors and combine of m + 1
    vectors into k + 1 outputs, CUDA events around `reps` launches after two warm-up launches; algorithmic bytes
    (m + 1 + k + 1) n 8 for blockDot, (m + 1 + k + 1) n 8 for combine (outputs written once).
  * A sequence of three right-hand sides (seeds 42, 44, 45) on one GCRODR(200, 30) handle, and a sequence of two
    factorizations: SetMatrix with the stored diagonal entries perturbed by 1e-3 relative (same pattern, as the
    driver's "Diagonal Perturbation") + Compute, then a solve that rebuilds C.
The card's name and power limit are read with nvidia-smi in the same run.
"""
import argparse
import copy
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import hymls_b200 as hb  # noqa: E402

SHIM = r'''
#include <cuda_runtime.h>
#include "kernels.hpp"
// ms of `reps` launches (which: 0 blockDot, 1 combine)
extern "C" int gt_time(int which, const double* X, int64_t n, int nx, const double* Y, int ny, double* partial,
                       double* H, int reps, float* ms) {
  try {
    cudaStream_t s = 0;
    int64_t launches = 0;
    auto one = [&]() {
      if (which == 0) hymls::blockDot(X, n, nx, Y, n, ny, n, partial, H, nx, s, &launches);
      else hymls::combine(X, n, nx, H, nx, const_cast<double*>(Y), n, ny, n, 0, s, &launches);
    };
    one();
    one();
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    cudaEventRecord(a, s);
    for (int r = 0; r < reps; ++r) one();
    cudaEventRecord(b, s);
    cudaEventSynchronize(b);
    cudaEventElapsedTime(ms, a, b);
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    return cudaGetLastError() == cudaSuccess ? 0 : -3;
  } catch (...) {
    return -1;
  }
}
extern "C" int64_t gt_partial() { return (int64_t)hymls::blockDotPartial(); }
'''
CONFIGS = [(100, 20), (200, 30), (300, 40)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def shim(tmp):
    lib_dir = os.path.dirname(hb.lib_path())
    cuda = os.environ.get("CUDA_HOME") or "/usr/local/cuda"
    src, so = os.path.join(tmp, "gt.cpp"), os.path.join(tmp, "gt.so")
    with open(src, "w") as f:
        f.write(SHIM)
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-I" + os.path.join(lib_dir, "csrc"),
                           "-I" + os.path.join(cuda, "include"), src, "-L" + lib_dir, "-lhymls_b200",
                           "-L" + os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + lib_dir,
                           "-Wl,-rpath," + os.path.join(cuda, "lib64"), "-o", so])
    lib = C.CDLL(so)
    lib.gt_time.argtypes = [C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                            C.c_int, C.POINTER(C.c_float)]
    lib.gt_partial.restype = C.c_int64
    return lib


def kernel_rates(lib, n, reps):
    import torch
    out = {}
    for m, k in CONFIGS:
        X = torch.empty((m + 1) * n, dtype=torch.float64, device="cuda").uniform_(-1, 1)
        Y = torch.empty((k + 1) * n, dtype=torch.float64, device="cuda").uniform_(-1, 1)
        H = torch.full(((m + 1) * (k + 1),), 1e-3, dtype=torch.float64, device="cuda")
        partial = torch.empty(lib.gt_partial(), dtype=torch.float64, device="cuda")
        for which, name in ((0, "blockDot"), (1, "combine")):
            ms = C.c_float()
            rc = lib.gt_time(which, X.data_ptr(), n, m + 1, Y.data_ptr(), k + 1, partial.data_ptr(), H.data_ptr(),
                             reps, C.byref(ms))
            assert rc == 0, rc
            per = ms.value / reps
            nbytes = (m + 1 + k + 1) * n * 8
            out["%s m+1=%d k+1=%d" % (name, m + 1, k + 1)] = {"ms": per, "tb_per_s": nbytes / (per * 1e-3) / 1e12,
                                                              "bytes": nbytes}
            print(name, m, k, "%.3f ms %.2f TB/s" % (per, nbytes / (per * 1e-3) / 1e12), flush=True)
        del X, Y, H, partial
        torch.cuda.empty_cache()
    return out


def run(P, b, x0):
    S = hb.Solver(P)
    x = S.ApplyInverse(b, x0.copy(), history_cap=8192)
    st = P.Stats()
    return {"iterations": S.num_iter, "converged": bool(S.info["converged"]), "solve_seconds": S.info["solve_seconds"],
            "explicit_rel_residual": S.info["explicit_rel_residual"], "krylov_basis_bytes": st["krylov_basis_bytes"],
            "krylov_recycle_dim": st["krylov_recycle_dim"], "num_apply_inverse": st["num_apply_inverse"]}, x


def handle(params, A, tv, method, m, k=None):
    p = copy.deepcopy(params)
    it = p["Solver"]["Iterative Solver"]
    p["Solver"]["Krylov Method"] = method
    if method == "GCRODR":
        it.update({"Num Blocks": m, "Num Recycled Blocks": k, "Maximum Restarts": 50, "Maximum Iterations": 5000})
    P = hb.Preconditioner(A, p, tv)
    P.Initialize()
    P.Compute()
    return P


def markdown(out):
    lines = ["# GCRO-DR against GMRES(600) on the bench problem", "",
             "Generated by `tools/gcrodr_timing.py` up to the Findings section, which is written by hand.", "",
             "`python tools/gcrodr_timing.py` on one %s (name, power limit), Stokes-C %d^3 (n = %d), skew partitioner, "
             "sx = 8, cx = 4, 2 levels, Right preconditioning, tolerance 1e-8 (Norm of Initial Residual). Raw numbers: "
             "`profiles/r08_gcrodr_1gpu.json`." % (out["card"], out["nx"], out["n"]), "",
             "| solver | iterations | converged | solve s | explicit residual | basis GB | recycled |",
             "|---|---|---|---|---|---|---|"]
    for key, r in out["solves"].items():
        lines.append("| %s | %d | %s | %.2f | %.2e | %.1f | %d |" % (
            key, r["iterations"], r["converged"], r["solve_seconds"], r["explicit_rel_residual"],
            r["krylov_basis_bytes"] / 1e9, r["krylov_recycle_dim"]))
    lines += ["", "Restart-phase kernels at n = %d (one launch each, bytes = (m + 1 + k + 1) n 8):" % out["n"], "",
              "| kernel | ms | TB/s |", "|---|---|---|"]
    for key, r in out["kernels"].items():
        lines.append("| %s | %.3f | %.2f |" % (key, r["ms"], r["tb_per_s"]))
    lines += ["", "Sequences on one GCRODR(200, 30) handle:", "", "| solve | iterations | solve s | recycled |",
              "|---|---|---|---|"]
    for key, r in out["sequences"].items():
        lines.append("| %s | %d | %.2f | %d |" % (key, r["iterations"], r["solve_seconds"], r["krylov_recycle_dim"]))
    return "\n".join(lines) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=128)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_gcrodr_1gpu.json"))
    ap.add_argument("--md", default=os.path.join(ROOT, "profiles", "r08_gcrodr.md"))
    args = ap.parse_args()
    import torch
    torch.cuda.set_device(0)
    params = bench.make_params(args.nx, 8, 2, 4)
    A, tv, _, b, x0 = bench.problem(args.nx)
    n = A.shape[0]
    with tempfile.TemporaryDirectory() as tmp:
        rates = kernel_rates(shim(tmp), n, args.reps)
    solves = {}
    P = handle(params, A, tv, "GMRES", 600)
    solves["GMRES(600)"], _ = run(P, b, x0)
    print("GMRES(600)", solves["GMRES(600)"], flush=True)
    del P
    torch.cuda.synchronize()
    for m, k in CONFIGS:
        P = handle(params, A, tv, "GCRODR", m, k)
        key = "GCRODR(%d, %d)" % (m, k)
        solves[key], _ = run(P, b, x0)
        print(key, solves[key], flush=True)
        del P
        torch.cuda.synchronize()
    seq = {}
    P = handle(params, A, tv, "GCRODR", 200, 30)
    for j, seed in enumerate((42, 44, 45)):
        bj = A @ np.random.default_rng(seed).uniform(-1, 1, n)
        seq["right-hand side %d" % (j + 1)], _ = run(P, bj, x0)
        print("rhs", j + 1, seq["right-hand side %d" % (j + 1)], flush=True)
    A2 = A.tocsr(copy=True)   # stored diagonal entries scaled by 1 + 1e-3 uniform(-1, 1): the same pattern
    rows = np.repeat(np.arange(n), np.diff(A2.indptr))
    on_diag = A2.indices == rows
    A2.data[on_diag] *= 1.0 + 1e-3 * np.random.default_rng(7).uniform(-1, 1, int(on_diag.sum()))
    P.SetMatrix(A2)
    P.Compute()
    seq["second factorization (C rebuilt)"], _ = run(P, A2 @ np.random.default_rng(46).uniform(-1, 1, n), x0)
    print("second factorization", seq["second factorization (C rebuilt)"], flush=True)
    del P
    out = {"card": card(), "n": int(n), "nx": args.nx, "sx": 8, "cx": 4, "levels": 2, "partitioner": bench.PARTITIONER,
           "reps": args.reps, "kernels": rates, "solves": solves, "sequences": seq}
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if args.md:
        findings = ""
        if os.path.exists(args.md):
            with open(args.md) as f:
                text = f.read()
            if "\n## Findings" in text:
                findings = text[text.index("\n## Findings"):]
        with open(args.md, "w") as f:
            f.write(markdown(out) + findings)


if __name__ == "__main__":
    main()
