"""Krylov solves on distributed vectors: hymls_b200_solve_dist (the rows of hymls_b200_owned_rows) and
hymls_b200_solve_map (the caller's row map), Solver.ApplyInverseDist / ApplyInverseMap, bordered right-hand sides
[b; T], and the Trilinos-side HYMLS::B200Solver (include/HYMLS_B200_Solver.hpp, driven by tests/solver_adapter_main.cpp).

The new entry points differ from hymls_b200_solve only in where b, x and the initial guess come from and go to, so on
one GPU and on every rank of a multi-GPU run they must reproduce its solution, iteration count and residual history
bit for bit.  Multi-rank cases run on 2 ranks, and on 4 when four devices are visible: one spawned process per GPU, a
gloo group for the NCCL id and for comparing results, NCCL inside the library.
"""
import ctypes as C
import os
import socket
import subprocess
import traceback

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

import hymls_b200 as hb
from hymls_b200 import driver

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_ARG, ERR_STATE, ERR_CUDA, ERR_UNSUPPORTED = -1, -2, -3, -99
EXPLICIT_FACTOR = 10.0   # explicit bordered residual <= this * Convergence Tolerance (right-preconditioned GMRES)


def _dictify(p):
    return {k: (_dictify(v) if isinstance(v, dict) else v) for k, v in p.items()}


def _solver(method="GMRES", side="Right", start="Zero", tol=1e-8, its=300):
    return {"Krylov Method": method, "Initial Vector": start, "Left or Right Preconditioning": side,
            "Iterative Solver": {"Maximum Iterations": its, "Num Blocks": its, "Maximum Restarts": 1,
                                 "Convergence Tolerance": tol}}


def _problem(name):
    """(params dict without "Solver", A, b, V or None) of the test problems"""
    from tests.common import make_params
    from tests.conftest import load_fixture
    if name == "cavity2d":
        A, b, _ = load_fixture("cavity2d_32_Re0")
        return _dictify(make_params("Stokes-C", 2, 32, 4, 2)), A, b, None
    if name == "stokes3d":   # the 3D case of test_gpu_parity.test_reference_3d_targets_with_skew_partitioner
        A, b, _ = load_fixture("cavity3d_16_Re0")
        return _dictify(make_params("Stokes-C", 3, 16, 8, 1, Partitioner="Skew Cartesian")), A, b, None
    assert name == "cavity.xml"  # configs/cavity.xml: bordered (Constant P), 3 levels, the Re 1000 fixture it names
    p = driver.parse_parameter_list(open(os.path.join(ROOT, "configs", "cavity.xml")).read())
    d = p.pop("Driver")
    A, b, _ = driver.read_system(d["Data Directory"])
    p.pop("Solver")
    return p, sp.csr_matrix(A), b, driver.create_nullspace(A.shape[0], d["Null Space Type"], p["Problem"])


def _build(name, solver, comm=None, border=True):
    p, A, b, V = _problem(name)
    p = dict(p)
    p["Solver"] = solver
    P = hb.Preconditioner(A, p, hb.galeri.create_testvector(A))
    if comm is not None:
        P.CommInit(*comm)
    P.Initialize()
    if border and V is not None:
        P.SetBorder(V)
    P.Compute()
    return P, A, b, V


def _bits(a):
    a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _same(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _c(x):
    return None if x is None else x.ctypes.data


def _raw(P, fn, b, T, x, S, where=hb.api.HOST):
    info = hb.api._SolveInfo()
    return getattr(P._lib, fn)(P._h, _c(b), _c(T), _c(x), _c(S), where, 43, C.byref(info), None, 0)


# ---------------------------------------------------------------------------------------------------------------
# no device
# ---------------------------------------------------------------------------------------------------------------
def test_entry_points_resolve_and_refuse_without_a_device():
    lib = hb.load_library()
    assert hasattr(lib, "hymls_b200_solve_dist") and hasattr(lib, "hymls_b200_solve_map")
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p, A, _, _ = _problem("cavity2d")
    p["Solver"] = _solver()
    P = hb.Preconditioner(A, p, pattern_only=True)
    P.Initialize()
    n = A.shape[0]
    for fn in ("hymls_b200_solve_dist", "hymls_b200_solve_map"):
        b, T = np.ones(n), np.ones(1)
        x, S = np.full(n, 7.0), np.full(1, 7.0)
        assert _raw(P, fn, b, T, x, S) == ERR_CUDA
        assert "needs a CUDA device" in P._lib.hymls_b200_last_error().decode()
        assert np.all(x == 7.0) and np.all(S == 7.0)


def _write_problem(tmp_path, nx):
    A = sp.csr_matrix(-hb.galeri.create_matrix("Stokes-C", 2, nx))
    A.sort_indices()
    tv = hb.galeri.create_testvector(A)
    mat, tvf = str(tmp_path / "A.bin"), str(tmp_path / "tv.bin")
    with open(mat, "wb") as f:
        np.asarray([A.shape[0], A.nnz, nx], dtype=np.int32).tofile(f)
        A.indptr.astype(np.int32).tofile(f)
        A.indices.astype(np.int32).tofile(f)
        A.data.astype(np.float64).tofile(f)
    tv.astype(np.float64).tofile(tvf)
    return A, tv, mat, tvf


def _build_driver(tmp_path):
    exe = str(tmp_path / "solver_adapter_main")
    lib_dir = os.path.dirname(hb.lib_path())
    cmd = ["/usr/bin/g++", "-std=c++17", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "tests", "shim"),
           "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "solver_adapter_main.cpp"),
           "-L" + lib_dir, "-lhymls_b200", "-Wl,-rpath," + lib_dir, "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_solver_adapter_header_compiles_links_and_fails_loudly_without_a_gpu(tmp_path):
    exe = _build_driver(tmp_path)
    _, _, mat, tvf = _write_problem(tmp_path, 16)
    r = subprocess.run([exe, mat, "1", tvf, str(tmp_path / "x.bin")], capture_output=True, text=True)
    # with a GPU the run succeeds; without one the library refuses loudly (no CPU fallback behind the adapter)
    assert r.returncode in (0, 3), (r.returncode, r.stderr)
    if r.returncode == 3:
        assert "needs a CUDA device" in r.stderr


# ---------------------------------------------------------------------------------------------------------------
# one GPU
# ---------------------------------------------------------------------------------------------------------------
SOLVES = [(prob, method, side, start) for prob in ("cavity2d", "stokes3d")
          for method, side in (("GMRES", "Right"), ("GMRES", "Left"), ("CG", "Right"))
          for start in ("Zero", "Random", "Previous")]


@pytest.mark.gpu
@pytest.mark.parametrize("prob,method,side,start", SOLVES)
def test_one_gpu_entry_points_match_the_replicated_solve(prob, method, side, start):
    import torch
    # CG on these indefinite systems need not converge: a fixed number of steps is compared
    solver = _solver(method, side, start, its=40 if method == "CG" else 300)
    P, A, b, _ = _build(prob, solver)
    n = A.shape[0]
    x0 = np.random.default_rng(3).uniform(-1, 1, n)
    ref = hb.Solver(P)
    x_ref = ref.ApplyInverse(b, x=x0.copy())
    perm = np.random.default_rng(4).permutation(n)
    P.SetRowMap(perm)
    S = hb.Solver(P)
    for entry, rows in (("ApplyInverseDist", np.arange(n)), ("ApplyInverseMap", perm)):
        for dev in (False, True):
            bl, xl = b[rows].copy(), x0[rows].copy()
            if dev:
                bl, xl = torch.from_numpy(bl).cuda(), torch.from_numpy(xl).cuda()
            x = getattr(S, entry)(bl, x=xl)
            assert x is xl
            what = "%s %s" % (entry, "device" if dev else "host")
            assert _same(x, x_ref[rows]), what
            assert S.num_iter == ref.num_iter, what
            assert _same(S.history, ref.history), what
            assert _same(S.info["explicit_rel_residual"], ref.info["explicit_rel_residual"]), what


@pytest.fixture(scope="module")
def bordered():
    P, A, b, V = _build("cavity.xml", _solver(tol=1e-10, its=250))
    return P, A, b, V


@pytest.mark.gpu
def test_bordered_without_T_matches_the_replicated_solve(bordered):
    P, A, b, V = bordered
    n = A.shape[0]
    ref = hb.Solver(P)
    x_ref = ref.ApplyInverse(b)
    perm = np.random.default_rng(5).permutation(n)
    P.SetRowMap(perm)
    S = hb.Solver(P)
    x, s = S.ApplyInverseDist(b.copy())
    assert _same(x, x_ref) and S.num_iter == ref.num_iter and _same(S.history, ref.history)
    x, s2 = S.ApplyInverseMap(b[perm].copy())
    assert _same(x, x_ref[perm]) and S.num_iter == ref.num_iter and _same(S.history, ref.history)
    assert _same(s, s2)


@pytest.mark.gpu
def test_bordered_with_T_solves_the_bordered_system(bordered):
    import torch
    P, A, b, V = bordered
    n, m = V.shape
    tol = 1e-10
    T = np.array([0.7])
    S = hb.Solver(P)
    x, s = S.ApplyInverseDist(b.copy(), T=T.copy())
    assert S.info["converged"]
    rb = np.concatenate([b, T])
    r = np.concatenate([A @ x + V @ s, V.T @ x]) - rb
    res = np.linalg.norm(r) / np.linalg.norm(rb)
    print("bordered solve: %d its, explicit residual %.2e (library %.2e)" % (S.num_iter, res,
                                                                           S.info["explicit_rel_residual"]))
    assert res <= EXPLICIT_FACTOR * tol
    assert S.info["explicit_rel_residual"] <= EXPLICIT_FACTOR * tol
    # against a direct solve of [K V; V' 0]: forward error <= cond * relative residual (2x for the direct solve's own
    # rounding)
    Kb = sp.bmat([[A, sp.csr_matrix(V)], [sp.csr_matrix(V.T), None]]).tocsc()
    z = spla.spsolve(Kb, rb)
    cond = np.linalg.cond(Kb.toarray())
    err = np.linalg.norm(np.concatenate([x, s]) - z) / np.linalg.norm(z)
    print("vs direct solve: %.2e, cond %.2e, bound %.2e" % (err, cond, 2 * cond * res))
    assert err <= 2 * cond * res
    # the other entry point and device buffers give the same bits; S is written only with a border
    perm = np.random.default_rng(6).permutation(n)
    P.SetRowMap(perm)
    xm, sm = S.ApplyInverseMap(b[perm].copy(), T=T.copy())
    assert _same(xm, x[perm]) and _same(sm, s)
    xd, sd = S.ApplyInverseDist(torch.from_numpy(b).cuda(), T=torch.from_numpy(T).cuda())
    assert _same(xd, x) and _same(sd, s)


@pytest.mark.gpu
def test_refused_calls_leave_the_buffers_untouched(bordered):
    Pb, A, b, V = bordered
    n = A.shape[0]

    def bufs():
        return np.ones(n), np.ones(1), np.full(n, 7.0), np.full(1, 7.0)

    def refused(P, fn, code, drop=None):
        bb, T, x, S = bufs()
        args = {"b": bb, "T": T, "x": x, "S": S}
        if drop:
            args[drop] = None
        assert _raw(P, fn, args["b"], args["T"], args["x"], args["S"]) == code, (fn, drop)
        assert np.all(x == 7.0) and np.all(S == 7.0)

    for fn in ("hymls_b200_solve_dist", "hymls_b200_solve_map"):
        Pb.SetRowMap(np.arange(n))
        refused(Pb, fn, ERR_ARG, "b")
        refused(Pb, fn, ERR_ARG, "x")
    # CG with a border set is refused as by hymls_b200_solve
    Pc, _, _, _ = _build("cavity.xml", _solver("CG"))
    Pc.SetRowMap(np.arange(n))
    for fn in ("hymls_b200_solve_dist", "hymls_b200_solve_map"):
        refused(Pc, fn, ERR_UNSUPPORTED)
    # before Compute; solve_map before set_row_map
    p, A2, b2, _ = _problem("cavity2d")
    p["Solver"] = _solver()
    P0 = hb.Preconditioner(A2, p, hb.galeri.create_testvector(A2))
    P0.Initialize()
    n2 = A2.shape[0]
    for fn in ("hymls_b200_solve_dist", "hymls_b200_solve_map"):
        x = np.full(n2, 7.0)
        assert _raw(P0, fn, np.ones(n2), None, x, None) == ERR_STATE and np.all(x == 7.0)
    P0.Compute()
    x = np.full(n2, 7.0)
    assert _raw(P0, "hymls_b200_solve_map", np.ones(n2), None, x, None) == ERR_STATE and np.all(x == 7.0)
    with pytest.raises(hb.HymlsError):
        hb.Solver(P0).ApplyInverseMap(np.ones(n2))
    # without a border T and S are neither read nor written
    T, S = np.full(1, np.nan), np.full(1, 7.0)
    x = np.zeros(n2)
    assert _raw(P0, "hymls_b200_solve_dist", b2, T, x, S) == 0
    assert np.isfinite(x).all() and S[0] == 7.0
    x_ref = hb.Solver(P0).ApplyInverse(b2)
    assert _same(x, x_ref)


@pytest.mark.gpu
def test_python_arguments_are_checked(bordered):
    import torch
    P, A, b, V = bordered
    n = A.shape[0]
    S = hb.Solver(P)
    B, T = np.zeros(n), np.zeros(1)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    bad = [dict(b_local=B[:-1]), dict(b_local=B, T=np.zeros(2)), dict(b_local=B.astype(np.float32)),
           dict(b_local=np.zeros(2 * n)[::2]), dict(b_local=B.reshape(1, -1)), dict(b_local=B, T=dev(T)),
           dict(b_local=B, x=np.zeros(n + 1)), dict(b_local=B, x=np.zeros(n, dtype=np.float32)),
           dict(b_local=dev(B), T=T), dict(b_local=torch.zeros(n, dtype=torch.float64)),
           dict(b_local=dev(B).float()), dict(b_local=torch.zeros(2 * n, dtype=torch.float64, device="cuda")[::2]),
           dict(b_local=dev(np.zeros(n + 1))), dict(b_local=dev(B), x=dev(np.zeros(n - 1)))]
    P.SetRowMap(np.arange(n))
    for entry in ("ApplyInverseDist", "ApplyInverseMap"):
        for kw in bad:
            with pytest.raises((ValueError, TypeError)):
                getattr(S, entry)(**kw)


@pytest.mark.gpu
def test_solver_adapter_equals_solve_map_on_a_permuted_row_map(tmp_path):
    exe = _build_driver(tmp_path)
    A, tv, mat, tvf = _write_problem(tmp_path, 16)
    out = str(tmp_path / "x.bin")
    r = subprocess.run([exe, mat, "1", tvf, out], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr     # the driver checks B200Solver against solve_map on its own handle
    assert "solver adapter ok" in r.stdout
    n = A.shape[0]
    o = np.fromfile(out, dtype=np.float64)
    X, xb, B = o[:2 * n].reshape(2, n), o[2 * n:3 * n], o[3 * n:5 * n].reshape(2, n)
    s, its = o[5 * n], o[5 * n + 1:5 * n + 3]
    # the same problem, parameters and row map through the Python binding
    p = {"Problem": {"Equations": "Stokes-C", "Dimension": 2, "nx": 16, "ny": 16, "nz": 1},
         "Preconditioner": {"Separator Length": 4, "Number of Levels": 1},
         "Solver": {"Krylov Method": "GMRES", "Left or Right Preconditioning": "Right", "Initial Vector": "Random",
                    "Iterative Solver": {"Maximum Iterations": 300, "Num Blocks": 300, "Maximum Restarts": 1,
                                         "Convergence Tolerance": 1e-8}}}
    P = hb.Preconditioner(A, p, tv)
    P.Initialize()
    P.Compute()
    perm = (np.arange(n) * 7 + 3) % n
    P.SetRowMap(perm)
    S = hb.Solver(P)
    for j in range(2):
        x = S.ApplyInverseMap(B[j][perm].copy())
        assert _same(x, X[j][perm]), j
    assert S.num_iter == its[0]
    V = np.zeros((n, 1))
    V[2::3, 0] = 1.0 / np.sqrt(n // 3)
    P.SetBorder(V)
    P.Compute()
    x, sb = S.ApplyInverseMap(B[0][perm].copy(), T=np.array([0.5]))
    assert _same(x, xb[perm]) and _same(sb[0], s) and S.num_iter == its[1]


# ---------------------------------------------------------------------------------------------------------------
# two and four GPUs
# ---------------------------------------------------------------------------------------------------------------
MULTI = ["cavity2d", "cavity.xml"]


def _worker(rank, world, port, out, dist_off):
    if dist_off:
        os.environ["HYMLS_B200_DIST"] = "0"
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

        def gather(obj):
            lst = [None] * world
            dist.all_gather_object(lst, obj)
            return lst

        for name in (MULTI[:1] if dist_off else MULTI):
            P, A, b, V = _build(name, _solver(start="Random", tol=1e-10, its=250), (comm_id(), rank, world))
            n = A.shape[0]
            r = res.setdefault(name, {})
            rows = P.OwnedRows()
            # a scattered caller map of uneven sizes
            perm = np.random.default_rng(9).permutation(n)
            cuts = np.sort(np.random.default_rng(10).choice(np.arange(1, n), world - 1, replace=False))
            mine = np.split(perm, cuts)[rank].astype(np.int64)
            P.SetRowMap(mine)
            ref, S = hb.Solver(P), hb.Solver(P)

            def run(fn):
                s0 = P.Stats()
                y = fn()
                s1 = P.Stats()
                return y, s1["collective_bytes"] - s0["collective_bytes"]

            x_ref, r["bytes_solve"] = run(lambda: ref.ApplyInverse(b))
            ys, r["bytes_dist"] = run(lambda: S.ApplyInverseDist(b[rows].copy()))
            eq = S.num_iter == ref.num_iter and _same(S.history, ref.history)
            xd = ys[0] if V is not None else ys
            ys, r["bytes_map"] = run(lambda: S.ApplyInverseMap(b[mine].copy()))
            xm = ys[0] if V is not None else ys
            eq = eq and S.num_iter == ref.num_iter and _same(S.history, ref.history)
            r["x_dist_equal"] = all(gather(bool(_same(xd, x_ref[rows]))))
            r["x_map_equal"] = all(gather(bool(_same(xm, x_ref[mine]))))
            r["its_history_equal"] = all(gather(bool(eq)))
            r["its"] = ref.num_iter
            r["n_own"] = gather(int(len(rows)))
            r["n_local"] = gather(int(len(mine)))
            if V is not None:   # T != 0: S bitwise equal on every rank and for both entry points
                T = np.array([0.7])
                xd, sd = S.ApplyInverseDist(b[rows].copy(), T=T.copy())
                xm, sm = S.ApplyInverseMap(b[mine].copy(), T=T.copy())
                parts = gather((rows, xd, sd))
                r["s_equal_on_ranks"] = all(_same(q[2], sd) for q in parts) and all(gather(bool(_same(sm, sd))))
                xg = np.zeros(n)
                for rr, xx, _ in parts:
                    xg[rr] = xx
                r["x_map_T_equal"] = all(gather(bool(_same(xm, xg[mine]))))
                rb = np.concatenate([b, T])
                rr = np.concatenate([A @ xg + V @ sd, V.T @ xg]) - rb
                r["residual_T"] = float(np.linalg.norm(rr) / np.linalg.norm(rb))
            del P
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


def _spawn(world, dist_off):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    key = (world, dist_off)
    if key not in _RESULTS:
        ctx = mp.get_context("spawn")
        out = ctx.Queue()
        port = _free_port()
        procs = [ctx.Process(target=_worker, args=(r, world, port, out, dist_off)) for r in range(world)]
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
        _RESULTS[key] = res
    return _RESULTS[key]


@pytest.fixture(scope="module", params=[2, 4], ids=["2ranks", "4ranks"])
def runs(request):
    return _spawn(request.param, False)


@pytest.mark.gpu
@pytest.mark.parametrize("name", MULTI)
def test_multi_rank_entry_points_equal_the_replicated_solve(runs, name):
    r = runs[name]
    assert r["x_dist_equal"] and r["x_map_equal"] and r["its_history_equal"]
    if name == "cavity.xml":
        assert r["s_equal_on_ranks"] and r["x_map_T_equal"]
        assert r["residual_T"] <= EXPLICIT_FACTOR * 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize("name", MULTI)
def test_multi_rank_collective_traffic(runs, name):
    r = runs[name]
    print("%s: solve %d B, solve_dist %d B, solve_map %d B (rank 0)" % (name, r["bytes_solve"], r["bytes_dist"],
                                                                        r["bytes_map"]))
    # hymls_b200_solve all-gathers x at the end: max_own doubles per rank; solve_dist skips exactly that
    assert r["bytes_solve"] - r["bytes_dist"] >= 8 * max(r["n_own"])
    # solve_map adds the two grouped exchanges of the caller's rows: rank 0 sends at most its n_local entries and
    # receives at most its n_own rows in each
    assert r["bytes_map"] - r["bytes_dist"] <= 2 * 8 * (r["n_local"][0] + r["n_own"][0])


@pytest.mark.gpu
def test_multi_rank_entry_points_on_the_replicated_path():
    r = _spawn(2, True)["cavity2d"]
    assert r["x_dist_equal"] and r["x_map_equal"] and r["its_history_equal"]
