"""ApplyInverse and GMRES timing of the bordered 128^3 Stokes-C cavity on N GPUs.  Run with torchrun:

    torchrun --nproc-per-node N tools/mgpu_border_timing.py [reps]
    HYMLS_B200_DIST=0 torchrun --nproc-per-node N tools/mgpu_border_timing.py [reps]   # replicated path

Workload: configs/cavity3D_128.xml with Fix Pressure Level = false and the Constant-P null space as border (m = 1),
the singular cavity Jacobian HYMLS solves with a bordered system.  Times, with device-resident owned vectors and
CUDA events: the bordered ApplyInverse (hymls_b200_apply_inverse_bordered_dist), the unbordered one on the same
matrix (hymls_b200_apply_inverse_dist after removing the border) and bordered GMRES to 1e-8.  HYMLS_B200_DIST is
read once per process, so the replicated path is a separate run.  Rank 0 prints one JSON line with the card name
and power limit read in the same run.
"""
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hymls_b200 as hb  # noqa: E402
from hymls_b200 import driver  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return q


def time_calls(fn, reps):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 50
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
    params["Preconditioner"]["Fix Pressure Level"] = False
    problem = params["Problem"]
    K = -hb.galeri.create_matrix("Stokes-C", 3, problem["nx"], problem["ny"], problem["nz"])
    n = K.shape[0]
    P = hb.Preconditioner(K, params, hb.galeri.create_testvector(K))
    if world > 1:
        P.CommInit(bytes(idt.numpy().tobytes()), rank, world)
    P.Initialize()
    V = driver.create_nullspace(n, "Constant P", problem)
    P.SetBorder(V)
    P.Compute()
    rows = P.OwnedRows()
    rng = np.random.default_rng(0)
    b = rng.uniform(-1, 1, n)
    bl = torch.from_numpy(b[rows]).cuda()
    T = torch.tensor([0.5], dtype=torch.float64, device="cuda")
    st0 = P.Stats()
    P.ApplyInverseBorderedDist(bl, T)
    st1 = P.Stats()
    ms_bordered = time_calls(lambda: P.ApplyInverseBorderedDist(bl, T), reps)
    x_ex = rng.uniform(-1, 1, n)
    x_ex -= V[:, 0] * (V[:, 0] @ x_ex)
    rhs = torch.from_numpy(K @ x_ex).cuda()
    S = hb.Solver(P)
    S.ApplyInverse(rhs)
    gm = {"iterations": S.num_iter, "converged": bool(S.info["converged"]), "solve_s": S.info["solve_seconds"],
          "explicit_rel_residual": S.info["explicit_rel_residual"]}
    coarse_rows = len(P.GetMap(hb.api.MAP_VSUM, P.NumLevels() - 1))
    P.SetBorder(None)
    P.Compute()
    st2 = P.Stats()
    P.ApplyInverseDist(bl)
    st3 = P.Stats()
    ms_plain = time_calls(lambda: P.ApplyInverseDist(bl), reps)
    dist.barrier()
    if rank == 0:
        print(json.dumps({
            "gpus": world, "path": "replicated (HYMLS_B200_DIST=0)" if os.environ.get("HYMLS_B200_DIST") == "0" and
            world > 1 else ("owner" if world > 1 else "single GPU"),
            "card": card(), "n": int(n), "border_columns": 1, "coarse_rows_bordered": coarse_rows + 1,
            "levels": P.NumLevels(), "reps": reps,
            "apply_bordered_ms": round(ms_bordered, 4), "apply_unbordered_ms": round(ms_plain, 4),
            "apply_bordered_collective_bytes": st1["collective_bytes"] - st0["collective_bytes"],
            "apply_unbordered_collective_bytes": st3["collective_bytes"] - st2["collective_bytes"],
            "gmres_bordered": gm}), flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
