"""GCRO-DR ("Krylov Method" = "GCRODR") on one GPU: the restart-phase kernels on their own (tests/gcrodr_harness.cpp),
then solves end to end against the numpy restatement of tests/gcrodr_reference.py, recycling across solves of one
handle, the rebuild of C after a Compute, repeatability, and the entry points on distributed vectors."""
import copy
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

import hymls_b200 as hb
from tests.gcrodr_reference import gcrodr
from tests.test_gpu_kernels import Kernels, _h
from tests.test_gpu_krylov_basis import _case

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_DIR = os.path.dirname(hb.lib_path())
TOL = 1e-8
_vp, _i32, _i64 = C.c_void_p, C.c_int, C.c_int64
_TAIL = [_vp, C.POINTER(C.c_int64)]
WRAPPERS = {
    "gh_block_dot": [_vp, _i64, _i32, _vp, _i64, _i32, _i64, _vp, _vp, _i64] + _TAIL,
    "gh_combine": [_vp, _i64, _i32, _vp, _i64, _vp, _i64, _i32, _i64, _i32] + _TAIL,
}


@pytest.fixture(scope="module")
def kernels(tmp_path_factory):
    import torch
    out = tmp_path_factory.mktemp("gcrodr_harness")
    cuda = os.environ.get("CUDA_HOME") or "/usr/local/cuda"
    so = os.path.join(str(out), "gcrodr_harness.so")
    cmd = ["/usr/bin/g++", "-std=c++17", "-Wall", "-Werror", "-fPIC", "-shared",
           "-I" + os.path.join(LIB_DIR, "csrc"), "-I" + os.path.join(cuda, "include"),
           os.path.join(ROOT, "tests", "gcrodr_harness.cpp"),
           "-L" + LIB_DIR, "-lhymls_b200", "-L" + os.path.join(cuda, "lib64"), "-lcudart",
           "-Wl,-rpath," + LIB_DIR, "-Wl,-rpath," + os.path.join(cuda, "lib64"), "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = C.CDLL(so)
    for name, argtypes in WRAPPERS.items():
        getattr(lib, name).argtypes = argtypes
        getattr(lib, name).restype = C.c_int
    lib.gh_block_dot_partial.restype = C.c_int64
    torch.cuda.set_device(0)
    return Kernels(lib), lib.gh_block_dot_partial()


# ---------------------------------------------------------------------------------------------------------------
# kernels: small integers, so every product and sum is exact in FP64 and the results equal an int64 reference
# bitwise.  n around the row tile (128) and the grid (296 blocks of 128 rows), nx around the 128 vectors of one
# launch, ny around 8 / 16 / 32 outputs, odd leading dimensions.
# ---------------------------------------------------------------------------------------------------------------
NS = [1, 127, 128, 129, 296 * 128 + 1, 2 ** 20 + 3]
SHAPES = [(1, 1), (7, 5), (31, 8), (128, 9), (129, 16), (301, 17), (41, 32), (33, 33)]


def _ints(shape, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randint(-8, 9, shape, device="cuda", generator=g, dtype=torch.int64)


@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("nx,ny", SHAPES)
def test_block_dot_is_exact(kernels, n, nx, ny):
    import torch
    kb, npart = kernels
    if n > 2 ** 17 and nx * ny > 300:
        pytest.skip("the largest n runs with the smaller shapes")
    ldx, ldy = n + 3, n | 1
    Xi, Yi = _ints((nx, ldx), n + nx), _ints((ny, ldy), 7 * n + ny)
    ref = (Xi[:, None, :n] * Yi[None, :, :n]).sum(dim=2).T.cpu().numpy().astype(np.float64)   # (ny, nx)
    partial = torch.full((npart,), float("nan"), dtype=torch.float64, device="cuda")
    ldh = nx + 2
    H = torch.full((ny * ldh,), float("nan"), dtype=torch.float64, device="cuda")
    kb("gh_block_dot", Xi.double(), ldx, nx, Yi.double(), ldy, ny, n, partial, H, ldh)
    got = _h(H).reshape(ny, ldh)
    assert np.array_equal(got[:, :nx], ref)
    assert np.all(np.isnan(got[:, nx:]))                           # nothing beyond nx is written


@pytest.mark.parametrize("accumulate", [0, 1])
@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("nx,ny", SHAPES)
def test_combine_is_exact(kernels, n, nx, ny, accumulate):
    kb, _ = kernels
    if n > 2 ** 17 and nx * ny > 300:
        pytest.skip("the largest n runs with the smaller shapes")
    ldx, ldy, ldc = n | 1, n + 5, nx + 1
    Xi, Ci, Yi = _ints((nx, ldx), n + 3 * nx), _ints((ny, ldc), nx + ny), _ints((ny, ldy), n + ny)
    ref = Yi.clone()                                       # entries beyond n stay as they were
    prod = (Ci[:, :nx, None] * Xi[None, :, :n]).sum(dim=1)
    ref[:, :n] = prod + (Yi[:, :n] if accumulate else 0)
    Y = Yi.double()
    kb("gh_combine", Xi.double(), ldx, nx, Ci.double(), ldc, Y, ldy, ny, n, accumulate)
    assert np.array_equal(_h(Y), ref.double().cpu().numpy())


def test_kernels_are_deterministic(kernels):
    import torch
    kb, npart = kernels
    n, nx, ny = 300_001, 200, 20
    g = torch.Generator(device="cuda").manual_seed(3)
    X = torch.randn((nx, n), device="cuda", generator=g, dtype=torch.float64)
    Y = torch.randn((ny, n), device="cuda", generator=g, dtype=torch.float64)
    coef = torch.randn((ny, nx), device="cuda", generator=g, dtype=torch.float64)
    out = []
    for _ in range(2):
        partial = torch.zeros(npart, dtype=torch.float64, device="cuda")
        H = torch.zeros(nx * ny, dtype=torch.float64, device="cuda")
        kb("gh_block_dot", X, n, nx, Y, n, ny, n, partial, H, nx)
        Z = torch.zeros((ny, n), dtype=torch.float64, device="cuda")
        kb("gh_combine", X, n, nx, coef, nx, Z, n, ny, n, 0)
        out.append((_h(H), _h(Z)))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
    ref = (Y.cpu().numpy() @ X.cpu().numpy().T)
    assert np.allclose(out[0][0].reshape(ny, nx), ref, rtol=1e-12, atol=1e-9)


# ---------------------------------------------------------------------------------------------------------------
# end to end against the reference
# ---------------------------------------------------------------------------------------------------------------
def _params(p, method="GCRODR", side="Right", blocks=30, k=5, restarts=100, its=2000, start="Zero"):
    q = copy.deepcopy(p)
    sol = q.setdefault("Solver", {})
    sol["Krylov Method"] = method
    sol["Left or Right Preconditioning"] = side
    sol["Initial Vector"] = start
    it = sol.setdefault("Iterative Solver", {})
    it.update({"Maximum Iterations": its, "Num Blocks": blocks, "Maximum Restarts": restarts,
               "Convergence Tolerance": TOL})
    if method == "GCRODR":
        it["Num Recycled Blocks"] = k
    else:
        it.pop("Num Recycled Blocks", None)
    return q


def _handle(p, A, V, **kw):
    P = hb.Preconditioner(A, _params(p, **kw), hb.galeri.create_testvector(A))
    P.Initialize()
    if V is not None:
        P.SetBorder(V, V, np.zeros((V.shape[1], V.shape[1])))
    P.Compute()
    return P


def _solve(P, b, entry="solve"):
    S = hb.Solver(P)
    if P.BorderSize() or entry != "solve":
        rows = P.OwnedRows()
        if entry == "map":
            P.SetRowMap(rows)
            fn = S.ApplyInverseMap
        else:
            fn = S.ApplyInverseDist
        n = len(b) - P.BorderSize()
        if P.BorderSize():
            xl, s = fn(b[:n][rows].copy(), b[n:].copy())
        else:
            xl, s = fn(b[rows].copy()), np.zeros(0)
        x = np.zeros(n)
        x[rows] = xl
        return S, np.concatenate([x, s])
    return S, S.ApplyInverse(b)


def _ops(P, A, V):
    """(A, M) of the solved system for the reference"""
    if V is None:
        return (lambda v: A @ v), P.ApplyInverse
    n = A.shape[0]

    def Ab(v):
        return np.concatenate([A @ v[:n] + V @ v[n:], V.T @ v[:n]])

    def M(v):
        X, Sv = P.ApplyInverseBordered(v[:n], v[n:])
        return np.concatenate([np.ravel(X), np.ravel(Sv)])
    return Ab, M


def _rhs(A, V, seed):
    rng = np.random.default_rng(seed)
    b = A @ rng.uniform(-1, 1, A.shape[0])
    return b if V is None else np.concatenate([b, np.zeros(V.shape[1])])


def _ref(P, A, V, b, side, blocks, k, U0=None, C0=None, info=None, reduction="qz"):
    Aop, M = _ops(P, A, V)
    return gcrodr(Aop, b, np.zeros(len(b)), apply_M=M, side=side, tol=TOL, max_iters=2000, num_blocks=blocks,
                  num_recycled=k, max_restarts=100, U0=U0, C0=C0, info=info, reduction=reduction)


def _rel_diff(h, ref, lo, hi):
    hi = min(hi, len(h), len(ref))
    if hi <= lo:
        return 0.0
    h, ref = np.asarray(h[lo:hi]), np.asarray(ref[lo:hi])
    return float(np.max(np.abs(h - ref) / np.abs(ref)))


# A recycled space is well determined only when its selection is separated from the harmonic Ritz values left out:
# with a relative gap (|theta_out| - |theta_in|) / |theta_in| below GAP_MIN, two correct implementations may keep
# different (equally valid) vectors, and the histories of the following cycles may differ by more than rounding.
GAP_MIN = 1e-3
# Even with clear gaps the harmonic problem itself can be sensitive.  The reference solves it three ways (QZ on the
# pencil, the Cholesky reduction of the library, the reduction by the QR factor of Ghat); when those disagree with each
# other, no implementation can be held closer to one of them than they are to each other.  Measured on a B200: with
# Right preconditioning the three agree to 1e-7 and the library to all of them; with Left preconditioning QZ and the
# reductions differ by up to 2.7e-3 (bordered64, k = 5) while the library stays within 2e-5 of the Cholesky and QR
# variants.  Later history entries are held to 1e-6 plus twice that spread.


CASES = ["stokes2d128", "skew16", "bordered64"]
BLOCKS = 40


@pytest.mark.parametrize("k", [1, 5, 20])
@pytest.mark.parametrize("side", ["Right", "Left"])
@pytest.mark.parametrize("name", CASES)
def test_against_the_reference(name, side, k):
    p, A, V = _case(name)
    P = _handle(p, A, V, side=side, blocks=BLOCKS, k=k)
    b = _rhs(A, V, 1)
    S, x = _solve(P, b)
    info = {}
    xr, itr, convr, hr, U, Cm = _ref(P, A, V, b, side, BLOCKS, k, info=info)
    h = S.history
    ends = info["cycle_ends"]
    # the first cycle is GMRES(m): the same history to 1e-10
    first = ends[0]
    assert np.max(np.abs(np.asarray(h[:first]) - np.asarray(hr[:first]))) <= 1e-10
    # later entries to 1e-6 relative, up to the first cycle that runs on a space selected across a gap < GAP_MIN
    strict = len(hr)
    for c, gap in info["gaps"]:
        if gap < GAP_MIN:
            strict = ends[c]
            break
    others = [_ref(P, A, V, b, side, BLOCKS, k, reduction=red)[3] for red in ("normal", "qr")]
    variants = [hr] + others
    spread = max(_rel_diff(u, v, first, strict) for i, u in enumerate(variants) for v in variants[i + 1:])
    per_cycle = ["%.1e" % _rel_diff(h, hr, lo, hi) for lo, hi in zip(ends[:-1], ends[1:])]
    to_variants = ["%.1e" % _rel_diff(h, v, first, strict) for v in others]
    print("%s %s k=%d: %d its (reference %d), recycled %d; selection gaps %s; history rel diff per later cycle %s; "
          "%d of %d entries compared; spread of the reference's reductions %.1e; library to normal / qr %s" % (
              name, side, k, S.num_iter, itr, P.Stats()["krylov_recycle_dim"],
              ["%.1e" % g for _, g in info["gaps"]], per_cycle, strict, len(hr), spread, to_variants))
    assert abs(S.num_iter - itr) <= 1
    assert _rel_diff(h, hr, first, strict) <= 1e-6 + 2 * spread
    assert strict >= min(len(hr), ends[1] if len(ends) > 1 else len(hr))  # at least the second cycle is compared
    assert S.info["converged"] == 1 and convr
    # converged = 1: the explicit residual in the implicit criterion's scaling (start vector zero) meets tol
    Aop, M = _ops(P, A, V)
    if side == "Right":
        assert np.linalg.norm(b - Aop(x)) / np.linalg.norm(b) <= TOL * 1.5
    else:
        assert np.linalg.norm(M(b - Aop(x))) / np.linalg.norm(M(b)) <= TOL * 1.5
    assert P.Stats()["krylov_recycle_dim"] in (k, k + 1)


@pytest.mark.parametrize("name", ["skew16", "bordered64"])
def test_three_right_hand_sides_on_one_handle(name):
    p, A, V = _case(name)
    k, blocks = 5, 30
    P = _handle(p, A, V, blocks=blocks, k=k)
    its, U, Cm = [], None, None
    for j in range(3):
        b = _rhs(A, V, 10 + j)
        calls = P.Stats()["num_apply_inverse"]
        S, x = _solve(P, b)
        calls = P.Stats()["num_apply_inverse"] - calls
        xr, itr, convr, hr, U, Cm = _ref(P, A, V, b, "Right", blocks, k, U0=U, C0=Cm)
        print("%s rhs %d: %d its (reference %d), %d ApplyInverse" % (name, j + 1, S.num_iter, itr, calls))
        assert abs(S.num_iter - itr) <= 1 and S.info["converged"]
        its.append(S.num_iter)
        # one ApplyInverse per iteration, one per cycle (the update of x), one for the projection of a recycled
        # solve; a rebuild of C would add k more
        kc = P.Stats()["krylov_recycle_dim"]
        cycles = -(-S.num_iter // (blocks - k - 1)) + 1
        assert S.num_iter < calls <= S.num_iter + cycles + (1 if j else 0)
    assert its[1] < its[0] and its[2] < its[0], its
    assert kc in (k, k + 1)


def test_set_matrix_rebuilds_c():
    p, A, V = _case("skew16")
    k, blocks = 5, 30
    P = _handle(p, A, V, blocks=blocks, k=k)
    b = _rhs(A, V, 20)
    S, _ = _solve(P, b)
    U = None
    _, _, _, _, U, Cm = _ref(P, A, V, b, "Right", blocks, k)
    # perturbed diagonal, as the driver's "Diagonal Perturbation"
    A2 = (A + sp.diags(1e-3 * np.random.default_rng(21).uniform(-1, 1, A.shape[0]) * abs(A.diagonal()))).tocsr()
    P.SetMatrix(A2)
    P.Compute()
    kc = P.Stats()["krylov_recycle_dim"]
    assert kc in (k, k + 1)                                          # SetMatrix + Compute keeps the space
    calls = P.Stats()["num_apply_inverse"]
    b2 = _rhs(A2, V, 22)
    S2, x2 = _solve(P, b2)
    calls = P.Stats()["num_apply_inverse"] - calls
    _, itr, convr, _, _, _ = _ref(P, A2, V, b2, "Right", blocks, k, U0=U)   # C rebuilt from U
    print("after SetMatrix: %d its (reference %d), %d ApplyInverse, %d recycled" % (S2.num_iter, itr, calls, kc))
    assert abs(S2.num_iter - itr) <= 1 and S2.info["converged"]
    assert calls >= S2.num_iter + kc + 1                              # the rebuild: kc operator applications
    assert np.linalg.norm(b2 - A2 @ x2) / np.linalg.norm(b2) <= TOL * 1.5


def test_two_handles_are_bitwise_equal():
    p, A, V = _case("skew16")
    out = []
    for _ in range(2):
        P = _handle(p, A, V, blocks=30, k=5, start="Random")
        runs = [_solve(P, _rhs(A, V, 30 + j)) for j in range(2)]
        out.append([(x, S.history) for S, x in runs])
    for a, b in zip(out[0], out[1]):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_gmres_after_gcrodr_equals_a_fresh_handle():
    p, A, V = _case("skew16")
    b = _rhs(A, V, 40)
    P = _handle(p, A, V, blocks=30, k=5)
    _solve(P, b)
    assert P.Stats()["krylov_recycle_dim"] > 0
    P.SetParameters(_params(p, method="GMRES", blocks=30))
    P.Initialize()
    P.Compute()
    assert P.Stats()["krylov_recycle_dim"] == 0
    S1, x1 = _solve(P, b)
    F = _handle(p, A, V, method="GMRES", blocks=30)
    S2, x2 = _solve(F, b)
    assert np.array_equal(x1, x2) and np.array_equal(S1.history, S2.history)
    # the GMRES solve freed U and the restart's scratch; the (grow-only) basis keeps the GCRODR size, k + 1 slots more
    assert P.Stats()["krylov_basis_bytes"] == 8 * (30 + 1 + 5 + 1) * A.shape[0]


@pytest.mark.parametrize("name", ["skew16", "bordered64"])
def test_recycle_dim_and_bytes(name):
    p, A, V = _case(name)
    m, k = 30, 7
    P = _handle(p, A, V, blocks=m, k=k)
    assert P.Stats()["krylov_recycle_dim"] == 0 and P.Stats()["krylov_basis_bytes"] == 0
    _solve(P, _rhs(A, V, 50))
    st = P.Stats()
    n = A.shape[0] + (0 if V is None else V.shape[1])
    assert st["krylov_recycle_dim"] in (k, k + 1)
    assert st["krylov_basis_bytes"] == 8 * (m + 1 + 3 * (k + 1)) * n
    P.Initialize()
    assert P.Stats()["krylov_recycle_dim"] == 0


@pytest.mark.parametrize("name", ["skew16", "bordered64"])
def test_distributed_entry_points_give_the_same_iterates(name):
    p, A, V = _case(name)
    out = {}
    for entry in ("solve", "dist", "map"):
        P = _handle(p, A, V, blocks=30, k=5)
        runs = [_solve(P, _rhs(A, V, 60 + j), entry) for j in range(2)]
        out[entry] = [(x, S.history) for S, x in runs]
    for entry in ("dist", "map"):
        for a, b in zip(out["solve"], out[entry]):
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_k_not_below_the_clamped_m_is_rejected_at_solve():
    p, A, V = _case("skew16")
    P = _handle(p, A, V, blocks=30, k=10, its=10)
    with pytest.raises(hb.HymlsError) as e:
        _solve(P, _rhs(A, V, 70))
    assert e.value.code == -1


# ---------------------------------------------------------------------------------------------------------------
# owner-distributed path on N ranks against one GPU (the pattern of test_gpu_krylov_basis.py): two solves per handle,
# the second one on the recycled space, a plain and a bordered case
# ---------------------------------------------------------------------------------------------------------------
def _worker(rank, world, port, out):
    import traceback
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    res = {}
    try:
        def comm_id():
            t = torch.zeros(128, dtype=torch.uint8)
            if rank == 0:
                t.copy_(torch.frombuffer(bytearray(hb.Preconditioner.CommUniqueId()), dtype=torch.uint8))
            dist.broadcast(t, 0)
            return bytes(t.numpy().tobytes())

        def gather(v):
            parts = [None] * world
            dist.all_gather_object(parts, v)
            return parts

        for name in ("skew16", "bordered64"):
            p, A, V = _case(name)
            n = A.shape[0]
            P = hb.Preconditioner(A, _params(p, blocks=30, k=5), hb.galeri.create_testvector(A))
            P.CommInit(comm_id(), rank, world)
            P.Initialize()
            if V is not None:
                P.SetBorder(V, V, np.zeros((V.shape[1], V.shape[1])))
            P.Compute()
            Q = _handle(p, A, V, blocks=30, k=5)          # one GPU, the same two solves
            rows = P.OwnedRows()
            runs = []
            for j in range(2):
                b = _rhs(A, V, 80 + j)
                S = hb.Solver(P)
                if V is not None:
                    xl, Sv = S.ApplyInverseDist(b[:n][rows].copy(), b[n:].copy())
                else:
                    xl, Sv = S.ApplyInverseDist(b[rows].copy()), np.zeros(0)
                parts = gather((rows, xl, Sv, P.Stats()["krylov_recycle_dim"]))
                x = np.zeros(n)
                for r_, x_, _, _ in parts:
                    x[r_] = x_
                x = np.concatenate([x, Sv])
                S1, x1 = _solve(Q, b)
                runs.append({"its": S.num_iter, "its_one_gpu": S1.num_iter, "converged": bool(S.info["converged"]),
                             "rel": float(np.linalg.norm(x - x1) / np.linalg.norm(x1)),
                             "S_equal": all(np.array_equal(s_, Sv) for _, _, s_, _ in parts),
                             "recycle_dims": [d for _, _, _, d in parts],
                             "recycle_dim_one_gpu": Q.Stats()["krylov_recycle_dim"]})
            res[name] = runs
            del P, Q
        ok = True
    except Exception:
        res = {"error": "rank %d: %s" % (rank, traceback.format_exc())}
        ok = False
    flags = torch.tensor([1 if ok else 0])
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    if rank == 0 or not ok:
        out.put(res)
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_owner_path_against_one_gpu(world):
    import torch
    import torch.multiprocessing as mp
    from tests.test_gpu_bordered_dist import _free_port
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        res = out.get(timeout=1500)
    finally:
        for p in procs:
            p.join(120)
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    assert "error" not in res, res.get("error")
    for name, runs in res.items():
        for j, r in enumerate(runs):
            print("%s solve %d on %d ranks: %d its (one GPU %d), x rel diff %.2e, recycled %s (one GPU %d)" % (
                name, j + 1, world, r["its"], r["its_one_gpu"], r["rel"], r["recycle_dims"],
                r["recycle_dim_one_gpu"]))
            assert r["converged"] and r["its"] == r["its_one_gpu"] and r["rel"] <= 1e-10 and r["S_equal"]
            assert len(set(r["recycle_dims"])) == 1 and r["recycle_dims"][0] == r["recycle_dim_one_gpu"] > 0
