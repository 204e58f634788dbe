"""End-to-end time of one GMRES solve through the three Krylov entry points, on N GPUs.  Run with torchrun:

    torchrun --nproc-per-node N tools/dist_solve_timing.py [out.json]

Workload: configs/cavity3D_128.xml (the bench.py problem: 128^3 Stokes-C, Skew Cartesian, sx = 8, cx = 4, 2 levels,
GMRES Right from zero to 1e-8, b = K x_ex with bench.py's x_ex).  One solve each, all with HOST vectors, as a
distributed Trilinos caller has them:
  * replicated: hymls_b200_solve, all n rows of b in and of x out on every rank;
  * dist:       hymls_b200_solve_dist on the rows of hymls_b200_owned_rows;
  * map:        hymls_b200_solve_map on a contiguous block row map (Epetra's default linear map).
An untimed solve first allocates the Krylov basis.  For every entry point the wall time from a barrier to the return
of the call (copies included; the maximum over the ranks) is reported beside the CUDA-event solve_seconds of the
Krylov loop and the collective bytes of rank 0.  Rank 0 prints one JSON line, with the card name and power limit read
in the same run, and writes it to out.json when given.
"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hymls_b200 as hb  # noqa: E402
from hymls_b200 import driver  # noqa: E402


def card():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                           str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()


def main():
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
    dist.init_process_group("gloo")
    idt = torch.zeros(128, dtype=torch.uint8)
    if rank == 0:
        idt.copy_(torch.frombuffer(bytearray(hb.Preconditioner.CommUniqueId()), dtype=torch.uint8))
    dist.broadcast(idt, 0)
    params = driver.parse_parameter_list(open(os.path.join(ROOT, "configs", "cavity3D_128.xml")).read())
    params.pop("Driver", None)
    problem = params["Problem"]
    K = -hb.galeri.create_matrix("Stokes-C", 3, problem["nx"], problem["ny"], problem["nz"])
    n = K.shape[0]
    P = hb.Preconditioner(K, params, hb.galeri.create_testvector(K))
    if world > 1:
        P.CommInit(bytes(idt.numpy().tobytes()), rank, world)
    P.Initialize()
    P.Compute()
    rows = P.OwnedRows()
    block = np.arange(rank * n // world, (rank + 1) * n // world, dtype=np.int64)
    P.SetRowMap(block)
    b = K @ np.random.default_rng(42).uniform(-1, 1, n)  # bench.py's right-hand side: a consistent system
    S = hb.Solver(P)
    S.ApplyInverse(b)  # allocates the Krylov basis
    runs = {}
    for name, call in (("replicated", lambda: S.ApplyInverse(b)),
                       ("dist", lambda: S.ApplyInverseDist(b[rows].copy())),
                       ("map", lambda: S.ApplyInverseMap(b[block].copy()))):
        st0 = P.Stats()
        dist.barrier()
        t0 = time.perf_counter()
        call()
        wall = torch.tensor([time.perf_counter() - t0], dtype=torch.float64)
        dist.all_reduce(wall, op=dist.ReduceOp.MAX)
        st1 = P.Stats()
        runs[name] = {"wall_s": round(float(wall[0]), 4), "solve_seconds": round(S.info["solve_seconds"], 4),
                      "iterations": S.num_iter, "converged": bool(S.info["converged"]),
                      "explicit_rel_residual": S.info["explicit_rel_residual"],
                      "collective_bytes_rank0": st1["collective_bytes"] - st0["collective_bytes"]}
    dist.barrier()
    if rank == 0:
        line = json.dumps({"gpus": world, "card": card(), "n": int(n), "n_owned_rank0": int(len(rows)),
                           "n_local_rank0": int(len(block)), "levels": P.NumLevels(), "vectors": "host",
                           "runs": runs})
        print(line, flush=True)
        if len(sys.argv) > 1:
            with open(sys.argv[1], "a") as f:
                f.write(line + "\n")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
