"""Double against Single "Krylov Basis Precision" on the bench problem, one GPU, in one process:

    python tools/krylov_basis_timing.py [--nx 128] [--reps 20] [--out FILE.json]

Kernel rates: the float and FP64 multiDot / multiAxpy launchers at n = 8 388 608 rows and k = 8, 64, 256, 600 basis
vectors, CUDA events around `reps` launches each after two warm-up launches, the two precisions alternated.  Algorithmic
bytes: k n sizeof(entry) + 8 n (w read) for the dot, k n sizeof(entry) + 16 n (w read and written) for the axpy.  Every
working set exceeds the 126 MB L2.  The launchers are reached through a small C++ shim compiled here into a temporary
directory against the in-tree library.

GMRES: the bench problem and inputs (Stokes-C 128^3, skew partitioner, sx = 8, cx = 4, 2 levels; b = A x_ex, x0
uniform(-1, 1) seed 43, GMRES(600) to 1e-8 in the "Norm of Initial Residual" scaling) for both basis precisions, each
with Double and with Single subdomain inverses, once with Maximum Restarts 0 (the bench) and once with 5.  Per run:
iterations, cycles, converged, solve_seconds, the explicit residual ||b - A x|| / ||b||, the FP64 residual after the
first cycle in the implicit scaling ||b - A x1|| / ||b - A x0|| (x1 from the Maximum Restarts 0 run), and the
krylov_basis_bytes and device_bytes of the handle.  The card's name and power limit are read in the same run.
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
// ms of `reps` launches of one launcher (which: 0 dot, 1 axpy; V32 != nullptr: the float basis)
extern "C" int kbt_time(int which, const double* V64, const float* V32, int64_t ldv, int k, double* w, int64_t n,
                        double* partial, double* h, int reps, float* ms) {
  try {
    cudaStream_t s = 0;
    int64_t launches = 0;
    auto one = [&]() {
      if (which == 0 && V32) hymls::multiDot(V32, ldv, k, w, n, partial, h, 0, s, &launches);
      else if (which == 0) hymls::multiDot(V64, ldv, k, w, n, partial, h, 0, s, &launches);
      else if (V32) hymls::multiAxpy(V32, ldv, k, h, w, n, 1.0, s, &launches);
      else hymls::multiAxpy(V64, ldv, k, h, w, n, 1.0, s, &launches);
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
'''


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def shim(tmp):
    lib_dir = os.path.dirname(hb.lib_path())
    cuda = os.environ.get("CUDA_HOME") or "/usr/local/cuda"
    src = os.path.join(tmp, "kbt.cpp")
    so = os.path.join(tmp, "kbt.so")
    with open(src, "w") as f:
        f.write(SHIM)
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-I" + os.path.join(lib_dir, "csrc"),
                           "-I" + os.path.join(cuda, "include"), src, "-L" + lib_dir, "-lhymls_b200",
                           "-L" + os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + lib_dir,
                           "-Wl,-rpath," + os.path.join(cuda, "lib64"), "-o", so])
    lib = C.CDLL(so)
    lib.kbt_time.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64, C.c_void_p,
                             C.c_void_p, C.c_int, C.POINTER(C.c_float)]
    return lib


def kernel_rates(lib, n, ks, reps):
    import torch
    kmax = max(ks)
    V64 = torch.empty(kmax * n, dtype=torch.float64, device="cuda")
    for i in range(kmax):
        V64[i * n:(i + 1) * n].uniform_(-1, 1)
    V32 = V64.float()
    w = torch.empty(n, dtype=torch.float64, device="cuda").uniform_(-1, 1)
    h = torch.full((kmax,), 1e-6, dtype=torch.float64, device="cuda")
    partial = torch.empty(kmax * 592, dtype=torch.float64, device="cuda")
    out = {}
    for k in ks:
        for which, name in ((0, "multiDot"), (1, "multiAxpy")):
            wbytes = 8 * n if which == 0 else 16 * n
            for prec in ("Double", "Single", "Double", "Single"):   # alternated; the second of each is reported too
                ms = C.c_float()
                rc = lib.kbt_time(which, V64.data_ptr() if prec == "Double" else None,
                                  V32.data_ptr() if prec == "Single" else None, n, k, w.data_ptr(), n,
                                  partial.data_ptr(), h.data_ptr(), reps, C.byref(ms))
                assert rc == 0, rc
                per = ms.value / reps
                nbytes = k * n * (8 if prec == "Double" else 4) + wbytes
                out.setdefault("%s k=%d" % (name, k), {}).setdefault(prec, []).append(
                    {"ms": per, "tb_per_s": nbytes / (per * 1e-3) / 1e12, "bytes": nbytes})
    del V64, V32
    torch.cuda.empty_cache()
    return out


def cycles(history, m, tol):
    """GMRES cycles of a run from its implicit residual history: a cycle ends after m steps or on the criterion"""
    c, k = 0, 0
    for rel in history[1:]:
        c += k == 0
        k += 1
        if rel <= tol or k == m:
            k = 0
    return c


def gmres_runs(params, A, tv, b, x0):
    import torch
    res = {}
    r0 = np.linalg.norm(b - A @ x0)
    for inv in ("Double", "Single"):
        for basis in ("Double", "Single"):
            for restarts in (0, 5):
                p = copy.deepcopy(params)
                p["Preconditioner"]["Subdomain Inverse Precision"] = inv
                p["Solver"]["Krylov Basis Precision"] = basis
                p["Solver"]["Iterative Solver"]["Maximum Restarts"] = restarts
                p["Solver"]["Iterative Solver"]["Maximum Iterations"] = 600 * (restarts + 1)
                P = hb.Preconditioner(A, p, tv)
                P.Initialize()
                P.Compute()
                S = hb.Solver(P)
                x = S.ApplyInverse(b, x0.copy(), history_cap=8192)
                st = P.Stats()
                key = "basis %s, inverses %s, Maximum Restarts %d" % (basis, inv, restarts)
                r = {"iterations": S.num_iter, "cycles": cycles(S.history, 600, 1e-8),
                     "converged": bool(S.info["converged"]), "solve_seconds": S.info["solve_seconds"],
                     "explicit_rel_residual": S.info["explicit_rel_residual"],
                     "implicit_rel_residual": S.info["rel_residual"],
                     "krylov_basis_bytes": st["krylov_basis_bytes"], "device_bytes": st["device_bytes"]}
                if restarts == 0:
                    r["first_cycle_fp64_residual"] = float(np.linalg.norm(b - A @ x) / r0)
                res[key] = r
                print(key, json.dumps(r), flush=True)
                del S, P
                torch.cuda.synchronize()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nx", type=int, default=128)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    torch.cuda.set_device(0)
    with tempfile.TemporaryDirectory() as tmp:
        lib = shim(tmp)
        rates = kernel_rates(lib, 8388608, [8, 64, 256, 600], args.reps)
    for key, v in rates.items():
        print(key, {p: ["%.3f ms %.2f TB/s" % (e["ms"], e["tb_per_s"]) for e in v[p]] for p in v}, flush=True)
    params = bench.make_params(args.nx, 8, 2, 4)
    A, tv, _, b, x0 = bench.problem(args.nx)
    gm = gmres_runs(params, A, tv, b, x0)
    out = {"card": card(), "n": int(A.shape[0]), "nx": args.nx, "sx": 8, "cx": 4, "levels": 2,
           "partitioner": bench.PARTITIONER, "kernel_n": 8388608, "reps": args.reps, "kernels": rates, "gmres": gm}
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
