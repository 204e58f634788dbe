"""Bordered systems on the owner-distributed multi-GPU path: hymls_b200_apply_inverse_bordered_dist /
Preconditioner.ApplyInverseBorderedDist, the bordered owner apply behind the replicated and caller-map entry points,
and bordered GMRES on the owner distribution, against single-GPU runs of the same inputs and the CPU oracle.

Every case runs on 2 ranks, and on 4 when four devices are visible: one spawned process per GPU, a gloo group for
the NCCL id and for comparing results, NCCL inside the library.

Accuracy of the multi-rank cases against single-GPU ApplyInverseBordered (asserted: ||X - X1|| / ||X1|| <= 1e-12,
||S - S1|| / ||S1|| <= 1e-10): not measured yet.  No run on two or more B200s has been recorded; on one GPU those cases
skip and only the one-rank and kernel tests below run.
"""
import ctypes as C
import os
import socket
import subprocess
import traceback

import numpy as np
import pytest
import scipy.sparse as sp

import hymls_b200 as hb

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_DIR = os.path.dirname(hb.lib_path())
TOL_X, TOL_S = 1e-12, 1e-10


def const_pressure(n, dof):
    V = np.zeros((n, 1))
    V[dof - 1::dof, 0] = 1.0
    return V / np.linalg.norm(V)


def _case(name):
    """(params, A, V, W, C, rhs, fixture) of the cases of test_gpu_bordered.py and a generated 32^3 cavity"""
    from tests.common import make_params
    from tests.conftest import load_fixture
    if name in ("bordering2", "m2-general"):
        A, b, _ = load_fixture("cavity2d_32_Re0")
        n = A.shape[0]
        if name == "bordering2":
            return make_params("Stokes-C", 2, 32, 4, 2, Fix_Pressure_Level=False), A, const_pressure(n, 3), None, None, b
        rng = np.random.default_rng(11)
        V = np.concatenate([const_pressure(n, 3), rng.uniform(-1, 1, (n, 1)) / np.sqrt(n)], axis=1)
        W = np.concatenate([rng.uniform(-1, 1, (n, 1)) / np.sqrt(n), const_pressure(n, 3)], axis=1)
        Cm = np.array([[0.5, -0.25], [0.125, 2.0]])
        return make_params("Stokes-C", 2, 32, 4, 3, 2), A, V, W, Cm, b
    if name == "3d-skew":
        A, b, _ = load_fixture("cavity3d_16_Re0")
        return (make_params("Stokes-C", 3, 16, 4, 2, 2, Partitioner="Skew Cartesian", Fix_Pressure_Level=False), A,
                const_pressure(A.shape[0], 4), None, None, b)
    assert name == "cube32-skew"
    A = sp.csr_matrix(-hb.galeri.create_matrix("Stokes-C", 3, 32))
    b = A @ np.random.default_rng(5).uniform(-1, 1, A.shape[0])
    return (make_params("Stokes-C", 3, 32, 8, 2, 2, Partitioner="Skew Cartesian", Fix_Pressure_Level=False), A,
            const_pressure(A.shape[0], 4), None, None, b)


CASES = ["bordering2", "m2-general", "3d-skew", "cube32-skew"]
# (case, side, start vector) of the bordered GMRES runs; m2-general (W != V, C != 0) has no V' x = 0 border row
SOLVES = [("bordering2", "Left", "Zero"), ("bordering2", "Left", "Random"), ("bordering2", "Right", "Zero"),
          ("bordering2", "Right", "Random"), ("3d-skew", "Right", "Zero"), ("3d-skew", "Left", "Random"),
          ("cube32-skew", "Right", "Random")]
FIXED_ITS = 20     # GMRES steps of the collective-traffic comparison


def _dictify(p):
    return {k: (_dictify(v) if isinstance(v, dict) else v) for k, v in p.items()}


def _solver(side, start, tol=1e-8, its=300, restarts=1):
    return {"Krylov Method": "GMRES", "Initial Vector": start, "Left or Right Preconditioning": side,
            "Iterative Solver": {"Maximum Iterations": its, "Num Blocks": its, "Maximum Restarts": restarts,
                                 "Convergence Tolerance": tol}}


def _build(p, A, V, W, Cm, solver, comm_id, rank, world, border=True):
    pd = _dictify(p)
    pd["Solver"] = solver
    P = hb.Preconditioner(A, pd, hb.galeri.create_testvector(A))
    if comm_id is not None:
        P.CommInit(comm_id, rank, world)
    P.Initialize()
    if border:
        P.SetBorder(V, W, Cm)
    P.Compute()
    return P


def _worker(rank, world, port, out):
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

        def allsum(v):
            t = torch.tensor(np.atleast_1d(np.asarray(v, dtype=np.float64)))
            dist.all_reduce(t)
            return t.numpy()

        def gather(obj):
            lst = [None] * world
            dist.all_gather_object(lst, obj)
            return lst

        for name in CASES:
            p, A, V, W, Cm, b = _case(name)
            n, m = V.shape
            r = res.setdefault(name, {"m": m})
            fixed = _solver("Right", "Zero", tol=1e-30, its=FIXED_ITS, restarts=0)
            P = _build(p, A, V, W, Cm, fixed, comm_id(), rank, world)
            Q = _build(p, A, V, W, Cm, fixed, None, rank, world)
            rows = P.OwnedRows()
            rng = np.random.default_rng(2)
            B = rng.uniform(-1, 1, n)
            T = rng.uniform(-1, 1, m)
            X1, S1 = Q.ApplyInverseBordered(B, T)
            X1, S1 = X1[:, 0], S1[:, 0]
            st0 = P.Stats()
            x, S = P.ApplyInverseBorderedDist(B[rows].copy(), T.copy())
            st1 = P.Stats()
            r["bordered_calls"] = st1["collective_calls"] - st0["collective_calls"]
            r["bordered_bytes"] = st1["collective_bytes"] - st0["collective_bytes"]
            num = allsum([np.sum((x - X1[rows]) ** 2), np.sum(X1[rows] ** 2)])
            r["x_rel"] = float(np.sqrt(num[0] / num[1]))
            r["s_rel"] = float(np.linalg.norm(S - S1) / np.linalg.norm(S1))
            r["s_equal_on_ranks"] = all(np.array_equal(s, S) for s in gather(S))
            # device buffers, and a second call: bitwise the same
            xd, Sd = P.ApplyInverseBorderedDist(torch.from_numpy(B[rows]).cuda(), torch.from_numpy(T).cuda())
            x2, S2 = P.ApplyInverseBorderedDist(B[rows].copy(), T.copy())
            r["repeat_equal"] = bool(np.array_equal(x2, x) and np.array_equal(S2, S) and
                                     np.array_equal(xd.cpu().numpy(), x) and np.array_equal(Sd.cpu().numpy(), S))
            # caller map = the owned rows, reversed: the same apply after a local permutation
            perm = rows[::-1].copy()
            P.SetRowMap(perm)
            Bm = np.asfortranarray(B[perm])
            Xm = np.zeros_like(Bm)
            Sm = np.zeros(m)
            hb.api._check(P._lib, P._lib.hymls_b200_apply_inverse_bordered_map(
                P._h, Bm.ctypes.data, len(perm), T.ctypes.data, Xm.ctypes.data, len(perm), Sm.ctypes.data, 1, hb.api.HOST))
            r["map_equal"] = bool(np.array_equal(Xm, x[::-1]) and np.array_equal(Sm, S))
            # the replicated bordered entry point runs the same owner apply
            Xr, Sr = P.ApplyInverseBordered(B, T)
            r["replicated_equal"] = bool(np.array_equal(Xr[rows, 0], x) and np.array_equal(Sr[:, 0], S))
            # ApplyInverseDist with a border set: T = 0, S discarded
            x0 = P.ApplyInverseDist(B[rows].copy())
            y1 = Q.ApplyInverse(B)
            num = allsum([np.sum((x0 - y1[rows]) ** 2), np.sum(y1[rows] ** 2)])
            r["t0_rel"] = float(np.sqrt(num[0] / num[1]))
            # the oracle (CPU, rank 0) on the gathered result
            if name != "cube32-skew":
                parts = gather((rows, x))
                if rank == 0:
                    from oracle import hymls as oh
                    Xg = np.zeros(n)
                    for rr, xx in parts:
                        Xg[rr] = xx
                    O = oh.Preconditioner(A, p.copy(), hb.galeri.create_testvector(A))
                    O.initialize()
                    O.set_border(V, W, Cm)
                    O.compute()
                    Xo, So = O.apply_inverse_bordered(B, T)
                    scale = np.linalg.norm(np.concatenate([Xo[:, 0], So[:, 0]]))
                    r["oracle_x"] = float(np.linalg.norm(Xg - Xo[:, 0]) / scale)
                    r["oracle_s"] = float(np.linalg.norm(S - So[:, 0]) / np.linalg.norm(So))
            # bordered GMRES with a fixed number of steps: collective traffic
            s0 = P.Stats()
            sol = hb.Solver(P)
            sol.ApplyInverse(b)
            s1 = P.Stats()
            r["gmres_its_bordered"] = sol.num_iter
            r["gmres_bytes_bordered"] = s1["collective_bytes"] - s0["collective_bytes"]
            r["levels"] = P.NumLevels()
            r["nS"] = int(P.Stats()["num_separator"])
            # the same matrix without the border: unbordered owner apply and GMRES
            P.SetBorder(None)
            P.Compute()
            s0 = P.Stats()
            P.ApplyInverseDist(B[rows].copy())
            s1 = P.Stats()
            r["plain_calls"] = s1["collective_calls"] - s0["collective_calls"]
            r["plain_bytes"] = s1["collective_bytes"] - s0["collective_bytes"]
            sol = hb.Solver(P)
            sol.ApplyInverse(b)
            s2 = P.Stats()
            r["gmres_its_plain"] = sol.num_iter
            r["gmres_bytes_plain"] = s2["collective_bytes"] - s1["collective_bytes"]
            del P, Q

        for name, side, start in SOLVES:
            p, A, V, W, Cm, b = _case(name)
            n = A.shape[0]
            solver = _solver(side, start)
            P = _build(p, A, V, W, Cm, solver, comm_id(), rank, world)
            Q = _build(p, A, V, W, Cm, solver, None, rank, world)
            S, S1 = hb.Solver(P), hb.Solver(Q)
            x = S.ApplyInverse(b)
            x1 = S1.ApplyInverse(b)
            k = min(len(S.history), len(S1.history), 15)
            res["%s/%s/%s" % (name, side, start)] = {
                "converged": bool(S.info["converged"]), "its": S.num_iter, "its_single": S1.num_iter,
                "hist_rel": float(np.max(np.abs(S.history[:k] - S1.history[:k]) / S1.history[:k])),
                "residual": float(np.linalg.norm(A @ x - b) / np.linalg.norm(b)),
                "vtx": float(abs(V[:, 0] @ x) / np.linalg.norm(x)),
                "x_equal_on_ranks": all(np.array_equal(v, x) for v in gather(x))}
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


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


_RESULTS = {}


@pytest.fixture(scope="module", params=[2, 4], ids=["2ranks", "4ranks"])
def runs(request):
    import torch
    import torch.multiprocessing as mp
    world = request.param
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    if world not in _RESULTS:
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
        assert all(p.exitcode == 0 for p in procs)
        _RESULTS[world] = res
    return _RESULTS[world]


@pytest.mark.parametrize("name", CASES)
def test_owner_apply_matches_single_gpu_and_oracle(runs, name):
    from tests.test_gpu_parity import TOL_STOKES
    r = runs[name]
    print("%s: X %.1e S %.1e T=0 %.1e" % (name, r["x_rel"], r["s_rel"], r["t0_rel"]))
    assert r["x_rel"] <= TOL_X and r["s_rel"] <= TOL_S
    assert r["t0_rel"] <= TOL_X          # ApplyInverseDist with a border = single-GPU ApplyInverse (T = 0)
    if "oracle_x" in r:
        assert r["oracle_x"] < TOL_STOKES and r["oracle_s"] < 1e-7


@pytest.mark.parametrize("name", CASES)
def test_owner_apply_is_reproducible_on_ranks_calls_and_entry_points(runs, name):
    r = runs[name]
    assert r["s_equal_on_ranks"]
    assert r["repeat_equal"]            # two calls, host and device buffers
    assert r["map_equal"]               # apply_inverse_bordered_map on a permuted caller map
    assert r["replicated_equal"]        # ApplyInverseBordered on replicated vectors


@pytest.mark.parametrize("name", CASES)
def test_border_adds_only_m_vectors_to_the_collectives(runs, name):
    r = runs[name]
    m = r["m"]
    extra_calls = r["bordered_calls"] - r["plain_calls"]
    extra = r["bordered_bytes"] - r["plain_bytes"]
    print("%s: apply %d calls / %d B bordered, %d / %d B plain" % (name, r["bordered_calls"], r["bordered_bytes"],
                                                                   r["plain_calls"], r["plain_bytes"]))
    assert 0 < extra_calls <= 2 * r["levels"] + 1
    assert extra <= 8 * m * extra_calls and extra <= 64 * m
    # the replicated fallback all-reduces two separator-length vectors: at least 16 nS bytes more
    assert extra < 16 * r["nS"]
    # GMRES: the same number of steps, the border costs O(m) doubles per step (operator + preconditioner)
    assert r["gmres_its_bordered"] == r["gmres_its_plain"] == FIXED_ITS
    per_it = (r["gmres_bytes_bordered"] - r["gmres_bytes_plain"]) / FIXED_ITS
    assert per_it <= 8 * m * (2 * r["levels"] + 4)


@pytest.mark.parametrize("key", ["%s/%s/%s" % s for s in SOLVES])
def test_bordered_gmres_on_the_owner_path(runs, key):
    r = runs[key]
    print("%s: %d its (single GPU %d), history %.1e, residual %.1e" % (key, r["its"], r["its_single"], r["hist_rel"],
                                                                      r["residual"]))
    assert r["converged"] and abs(r["its"] - r["its_single"]) <= 1
    assert r["hist_rel"] <= 1e-6
    assert r["residual"] <= 1e-6 and r["vtx"] <= 1e-6
    assert r["x_equal_on_ranks"]


# ---------------------------------------------------------------------------------------------------------------
# one rank: the entry point is hymls_b200_apply_inverse_bordered; arguments are checked before any device work
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def one_rank():
    p, A, V, W, Cm, _ = _case("m2-general")
    return _build(p, A, V, W, Cm, _solver("Right", "Zero"), None, 0, 1), A.shape[0]


def test_one_rank_equals_the_replicated_bordered_entry_point(one_rank):
    import torch
    P, n = one_rank
    assert P.BorderSize() == 2 and np.array_equal(P.OwnedRows(), np.arange(n))
    rng = np.random.default_rng(8)
    B, T = rng.uniform(-1, 1, n), rng.uniform(-1, 1, 2)
    X1, S1 = P.ApplyInverseBordered(B, T)
    x, S = P.ApplyInverseBorderedDist(B, T)
    assert np.array_equal(x, X1[:, 0]) and np.array_equal(S, S1[:, 0])
    xd, Sd = P.ApplyInverseBorderedDist(torch.from_numpy(B).cuda(), torch.from_numpy(T).cuda())
    assert np.array_equal(xd.cpu().numpy(), x) and np.array_equal(Sd.cpu().numpy(), S)


def test_bordered_dist_arguments_are_checked(one_rank):
    import torch
    P, n = one_rank
    B, T = np.zeros(n), np.zeros(2)
    bad = [(B[:-1], T), (B, np.zeros(3)), (B.astype(np.float32), T), (np.zeros(2 * n)[::2], T),
           (B.reshape(1, -1), T), (B, torch.zeros(2, dtype=torch.float64, device="cuda")),
           (torch.zeros(n, dtype=torch.float64, device="cuda"), T),
           (torch.zeros(n, dtype=torch.float64), torch.zeros(2, dtype=torch.float64)),
           (torch.zeros(n, dtype=torch.float32, device="cuda"), torch.zeros(2, dtype=torch.float64, device="cuda")),
           (torch.zeros(2 * n, dtype=torch.float64, device="cuda")[::2],
            torch.zeros(2, dtype=torch.float64, device="cuda")),
           (torch.zeros(n + 1, dtype=torch.float64, device="cuda"), torch.zeros(2, dtype=torch.float64, device="cuda"))]
    for b, t in bad:
        with pytest.raises((ValueError, TypeError)):
            P.ApplyInverseBorderedDist(b, t)


# ---------------------------------------------------------------------------------------------------------------
# the kernels, one at a time, on integer inputs (every sum exact: bitwise equal to the exact result)
# ---------------------------------------------------------------------------------------------------------------
_vp, _i32, _i64 = C.c_void_p, C.c_int, C.c_int64
_TAIL = [_vp, C.POINTER(C.c_int64)]
WRAPPERS = {
    "bdh_border_spmv_rows": [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _i64, _vp, _vp, _vp] + _TAIL,
    "bdh_multi_dot_rows": [_vp, _i64, _i32, _vp, _i64, _vp, _vp, _vp, _vp] + _TAIL,
    "bdh_border_correct_list": [_vp, _vp, _vp, _i64, _i32, _vp, _i64, _vp] + _TAIL,
    "bdh_multi_dot_blocks": [],
}


@pytest.fixture(scope="module")
def kh(tmp_path_factory):
    import torch
    cuda = os.environ.get("CUDA_HOME") or "/usr/local/cuda"
    so = os.path.join(str(tmp_path_factory.mktemp("bordered_dist_harness")), "bordered_dist_harness.so")
    cmd = ["/usr/bin/g++", "-std=c++17", "-Wall", "-Werror", "-fPIC", "-shared",
           "-I" + os.path.join(LIB_DIR, "csrc"), "-I" + os.path.join(cuda, "include"),
           os.path.join(ROOT, "tests", "bordered_dist_harness.cpp"),
           "-L" + LIB_DIR, "-lhymls_b200", "-L" + os.path.join(cuda, "lib64"), "-lcudart",
           "-Wl,-rpath," + LIB_DIR, "-Wl,-rpath," + os.path.join(cuda, "lib64"), "-o", so]
    rc = subprocess.run(cmd, capture_output=True, text=True)
    assert rc.returncode == 0, rc.stderr
    lib = C.CDLL(so)
    for fn, argtypes in WRAPPERS.items():
        getattr(lib, fn).argtypes = argtypes
        getattr(lib, fn).restype = C.c_int
    torch.cuda.set_device(0)
    return lib


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _call(kh, fn, *args):
    import torch
    launches = C.c_int64(0)
    rc = getattr(kh, fn)(*args, C.c_void_p(torch.cuda.current_stream().cuda_stream), C.byref(launches))
    assert rc == 0
    return launches.value


def _rand_csr(rng, n, per_row):
    nnz = rng.integers(0, per_row + 1, n)
    ptr = np.concatenate([[0], np.cumsum(nnz)]).astype(np.int64)
    col = rng.integers(0, n, int(ptr[-1])).astype(np.int32)
    val = rng.integers(-8, 9, int(ptr[-1])).astype(np.float64)
    return ptr, col, val


@pytest.mark.parametrize("m", [1, 2, 8, 9])
@pytest.mark.parametrize("nrows", [0, 1, 1000, 200_003])
def test_border_spmv_rows_is_exact(kh, m, nrows):
    rng = np.random.default_rng(100 * m + nrows % 97)
    n = max(2 * nrows, 16)
    ptr, col, val = _rand_csr(rng, n, 7)
    x = rng.integers(-64, 65, n).astype(np.float64)
    V = rng.integers(-16, 17, (m, n)).astype(np.float64)     # column j of the n x m border at V[j]
    W = rng.integers(-16, 17, (m, n)).astype(np.float64)
    sv = rng.integers(-16, 17, m).astype(np.float64)
    rows = rng.permutation(n)[:nrows].astype(np.int32)
    K = sp.csr_matrix((val, col, ptr), shape=(n, n))
    want_y = (K @ x + V.T @ sv)[rows]
    want_d = W[:, rows] @ x[rows]
    y = _dev(np.full(max(nrows, 1), np.nan))
    partial = _dev(np.full(m * kh.bdh_multi_dot_blocks(), np.nan))
    dots = _dev(np.full(m, np.nan))
    d = [_dev(a) for a in (ptr, col, val, x, V, W)]       # kept alive until the kernel has run
    dsv, drows = _dev(sv), _dev(rows)
    launches = _call(kh, "bdh_border_spmv_rows", *[a.data_ptr() for a in d[:4]], d[4].data_ptr(), d[5].data_ptr(),
                     n, m, dsv.data_ptr(), drows.data_ptr(), nrows, y.data_ptr(), partial.data_ptr(), dots.data_ptr())
    assert launches == 2
    assert np.array_equal(y.cpu().numpy()[:nrows], want_y)
    assert np.array_equal(dots.cpu().numpy(), want_d)


@pytest.mark.parametrize("k", [1, 2, 9])
@pytest.mark.parametrize("nlist", [0, 7, 300_001])
@pytest.mark.parametrize("gather", [False, True])
def test_multi_dot_on_a_row_list_is_exact(kh, k, nlist, gather):
    rng = np.random.default_rng(7 * k + nlist % 31 + gather)
    nv = max(nlist + nlist // 3, 8)
    V = rng.integers(-32, 33, (k, nv)).astype(np.float64)
    nw = nv + 5
    w = rng.integers(-32, 33, nw).astype(np.float64)
    widx = rng.permutation(nw)[:nv].astype(np.int32)
    rows = rng.permutation(nv)[:nlist].astype(np.int32)
    want = V[:, rows] @ (w[widx[rows]] if gather else w[rows])
    h = _dev(np.full(k, np.nan))
    partial = _dev(np.full(k * kh.bdh_multi_dot_blocks(), np.nan))
    dV, dw, dwidx, drows = _dev(V), _dev(w), _dev(widx), _dev(rows)
    _call(kh, "bdh_multi_dot_rows", dV.data_ptr(), nv, k, dw.data_ptr(), nlist, partial.data_ptr(), h.data_ptr(),
          dwidx.data_ptr() if gather else None, drows.data_ptr())
    assert np.array_equal(h.cpu().numpy(), want)


@pytest.mark.parametrize("m", [1, 3])
@pytest.mark.parametrize("nlist", [0, 5, 100_000])
def test_border_correct_on_a_position_list_is_exact(kh, m, nlist):
    rng = np.random.default_rng(13 * m + nlist)
    npos = max(2 * nlist, 8)
    nx = npos + 11
    X = rng.integers(-1000, 1001, nx).astype(np.float64)
    idx = rng.permutation(nx)[:npos].astype(np.int32)
    Q = rng.integers(-16, 17, (m, npos)).astype(np.float64)
    S = rng.integers(-16, 17, m).astype(np.float64)
    lst = rng.permutation(npos)[:nlist].astype(np.int32)
    want = X.copy()
    want[idx[lst]] -= S @ Q[:, lst]
    dX, didx, dQ, dS, dlst = _dev(X), _dev(idx), _dev(Q), _dev(S), _dev(lst)
    _call(kh, "bdh_border_correct_list", dX.data_ptr(), didx.data_ptr(), dQ.data_ptr(), npos, m, dS.data_ptr(), nlist,
          dlst.data_ptr())
    assert np.array_equal(dX.cpu().numpy(), want)       # positions outside the list untouched
