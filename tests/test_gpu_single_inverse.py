"""FP32 storage of the subdomain inverses ("Subdomain Inverse Precision" = "Single"): the float paths of the slab and
multi-vector GEMV kernels and the narrowing kernel on their own (tests/single_inverse_harness.cpp), then Double and
Single handles on the same matrices end to end, on one GPU and on the owner-distributed path with 2 or 4 ranks.

Accuracy of Single against Double: the tests assert ApplyInverse within SINGLE_TOL = 1e-5 relative (2^-24 with an
amplification allowance of about 170; not a derived bound) and print the measured values.  Measured on a B200:
2.2e-8 .. 4.2e-7 on the cases below, 7.9e-6 on the 128^3 bench problem (profiles/r05_single_inverse.md), so the
bound is kept as it is."""
import ctypes as C
import os
import subprocess
import traceback

import numpy as np
import pytest
import scipy.sparse as sp

import hymls_b200 as hb
from tests.test_gpu_kernels import (BATCHED_OPTS, GEMV_SHAPES, MULTI_OPTS, SENTINEL, GemvCase, Kernels, _build_harness,
                                    _d, _h)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_DIR = os.path.dirname(hb.lib_path())
SINGLE_TOL = 1e-5
ERR_STATE = -2

# ---------------------------------------------------------------------------------------------------------------
# kernels: the float launchers against the FP64 launchers on integer matrices (every product and sum exact, and every
# entry exact in FP32), hence bitwise equal.  np = 1032 (258 float4 per row) runs the 4-load unrolled loop of the slab
# kernel twice, 512 / 520 once, 264 and below only the remainder loop.
# ---------------------------------------------------------------------------------------------------------------
SHAPES = GEMV_SHAPES + [(1032, 1032), (1032, 1029)]
_vp, _i32, _i64 = C.c_void_p, C.c_int, C.c_int64
_GEMV = [_vp] * 16 + [_i32, _i32]
_TAIL = [_vp, C.POINTER(C.c_int64)]
WRAPPERS = {
    "sih_batched_gemv": _GEMV + [_i32, _i32] + _TAIL,
    "sih_batched_gemv_multi": _GEMV + [_i32, _i32, _i32, _i64, _i64, _i64, _vp] + _TAIL,
    "sih_batched_gemv_t": _GEMV + [_i32, _i32] + _TAIL,
    "sih_narrow_to_float": [_vp, _vp, _i64, _vp] + _TAIL,
}


@pytest.fixture(scope="module")
def kernels(tmp_path_factory):
    import torch
    out = tmp_path_factory.mktemp("single_inverse_harness")
    cuda = os.environ.get("CUDA_HOME") or "/usr/local/cuda"
    so = os.path.join(str(out), "single_inverse_harness.so")
    cmd = ["/usr/bin/g++", "-std=c++17", "-Wall", "-Werror", "-fPIC", "-shared",
           "-I" + os.path.join(LIB_DIR, "csrc"), "-I" + os.path.join(cuda, "include"),
           os.path.join(ROOT, "tests", "single_inverse_harness.cpp"),
           "-L" + LIB_DIR, "-lhymls_b200", "-L" + os.path.join(cuda, "lib64"), "-lcudart",
           "-Wl,-rpath," + LIB_DIR, "-Wl,-rpath," + os.path.join(cuda, "lib64"), "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = C.CDLL(so)
    for name, argtypes in WRAPPERS.items():
        getattr(lib, name).argtypes = argtypes
        getattr(lib, name).restype = C.c_int
    torch.cuda.set_device(0)
    return Kernels(lib), Kernels(_build_harness(out))


def _args32(c, d, A32, im, ir, nrows):
    args = list(c.gemv_args(d, im, ir, nrows))
    args[9] = A32
    return args


def _run_both(kernels, c, d, name64, name32, launch):
    """launch(kh, name, d, A) with the FP64 launcher and the float one on fresh output buffers; returns both outputs"""
    k32, k64 = kernels
    outs = []
    for kh, name, A in ((k64, name64, d["A"]), (k32, name32, _d(c.A.astype(np.float32)))):
        dd = dict(d)
        dd["out"] = _d(np.full(d["out"].numel(), SENTINEL))
        launch(kh, name, dd, A)
        outs.append(_h(dd["out"]))
    return outs


@pytest.mark.parametrize("opts", BATCHED_OPTS, ids=lambda o: "+".join(o) or "plain")
def test_float_slab_gemv_equals_fp64(kernels, opts):
    c = GemvCase(opts, seed=7 + len(opts), shapes=SHAPES)
    assert np.array_equal(c.A.astype(np.float32), c.A)
    d = c.device()
    npmax = int(c.np_.max())

    def launch(kh, name, dd, A):
        if c.nrows_lead is not None:   # lead items with nrows, then the trail items without it (ApplyInverse's split)
            lead = c.nrows_lead
            im, ir = c.items(last=lambda m: int(lead[m]))
            assert kh(name, *_args32(c, dd, A, _d(im), _d(ir), dd["nrows"]), len(im), npmax) == 1
            im, ir = c.items(first=lambda m: int(lead[m]))
            assert kh(name, *_args32(c, dd, A, _d(im), _d(ir), None), len(im), npmax) == 1
        else:
            im, ir = c.items()
            assert kh(name, *_args32(c, dd, A, _d(im), _d(ir), dd["nrows"]), len(im), npmax) == 1

    got64, got32 = _run_both(kernels, c, d, "kh_batched_gemv", "sih_batched_gemv", launch)
    assert np.array_equal(got64.reshape(1, -1), c.expected())
    assert np.array_equal(got32, got64)


@pytest.mark.parametrize("nv", [2, 3, 4])
@pytest.mark.parametrize("opts", MULTI_OPTS, ids=lambda o: "+".join(o) or "plain")
def test_float_multi_gemv_equals_fp64(kernels, nv, opts):
    c = GemvCase(opts, seed=2000 + 10 * nv + len(opts), shapes=SHAPES, nv=nv)
    d = c.device()
    npmax = int(c.np_.max())
    pad_in, pad_sub, pad_out = 5, 3, 9
    ld_in, ld_sub, ld_out = c.nin + pad_in, int(c.vecOff[-1]) + pad_sub, c.nout + pad_out
    xin = np.full((nv, ld_in), 7.0)
    xin[:, :c.nin] = c.xin
    d["xin"] = _d(xin.ravel())
    if c.xsub is not None:
        xs = np.full((nv, ld_sub), -3.0)
        xs[:, :ld_sub - pad_sub] = c.xsub
        d["xsub"] = _d(xs.ravel())
    d["out"] = _d(np.full(nv * ld_out, SENTINEL))
    if c.nrows_lead is not None:
        im, ir = c.items(last=lambda m: int(c.nrows_lead[m]))
    else:
        im, ir = c.items()

    def launch(kh, name, dd, A):
        accepted = C.c_int(0)
        assert kh(name, *_args32(c, dd, A, _d(im), _d(ir), dd["nrows"]), len(im), npmax, nv, ld_in, ld_sub,
                  ld_out, C.byref(accepted)) == 1
        assert accepted.value == 1

    got64, got32 = _run_both(kernels, c, d, "kh_batched_gemv_multi", "sih_batched_gemv_multi", launch)
    rows = (lambda m: (0, int(c.nrows_lead[m]))) if c.nrows_lead is not None else None
    assert np.array_equal(got64.reshape(nv, ld_out)[:, :c.nout], c.expected(rows=rows))
    assert np.all(got64.reshape(nv, ld_out)[:, c.nout:] == SENTINEL)
    assert np.array_equal(got32, got64)


def test_transposed_gemv_refuses_a_float_store(kernels):
    k32, _ = kernels
    c = GemvCase((), seed=3, shapes=[(16, 13)])
    d = c.device()
    launches = C.c_int64(0)
    import torch
    A32 = _d(c.A.astype(np.float32))
    rc = k32.lib.sih_batched_gemv_t(*[a.data_ptr() if isinstance(a, torch.Tensor) else a
                                      for a in _args32(c, d, A32, None, None, None)], 1, 16,
                                    torch.cuda.current_stream().cuda_stream, C.byref(launches))
    assert rc == ERR_STATE and launches.value == 0


def _narrow_values():
    rng = np.random.default_rng(5)
    f32max = float(np.finfo(np.float32).max)
    tiny = 2.0 ** -149                                  # smallest float subnormal
    specials = [0.0, -0.0, 1.0, -1.0, 1.0 + 2.0 ** -24, 1.0 + 3 * 2.0 ** -24, -(1.0 + 2.0 ** -24),   # ties
                2.0 ** -126, 2.0 ** -127 * 1.5, 1e-40, -1e-40, tiny, 1.5 * tiny, 2.5 * tiny, 0.5 * tiny,  # subnormals
                0.25 * tiny, 3e-46, f32max, -f32max, f32max * (1 + 2.0 ** -25), np.inf, -np.inf,
                np.pi, -np.e, 1e-300]
    v = np.concatenate([rng.standard_normal(100_000) * 10.0 ** rng.integers(-50, 38, 100_000),
                        (rng.integers(-2 ** 24, 2 ** 24, 20_000) + 0.5) * 2.0 ** rng.integers(-160, 100, 20_000)])
    v = v[np.abs(v) <= f32max]
    return np.concatenate([specials, v, specials[::-1]])


def _narrow(k32, src, chunks):
    """the engine's in-place narrowing: chunk [o0, o1) into a work buffer, then onto float index o0 of the store"""
    import torch
    store = _d(src)
    store32 = store.view(torch.float32)
    work = torch.full((int(np.max(np.diff(chunks))),), np.nan, dtype=torch.float32, device="cuda")
    flag = _d(np.zeros(1, dtype=np.int32))
    for o0, o1 in zip(chunks[:-1], chunks[1:]):
        k32("sih_narrow_to_float", store.data_ptr() + 8 * int(o0), work, int(o1 - o0), flag)
        store32[o0:o1].copy_(work[:o1 - o0])
    torch.cuda.synchronize()
    return _h(store32[:len(src)]), int(_h(flag)[0])


@pytest.mark.parametrize("chunking", ["one", "split_matrices", "tiny"])
def test_narrowing_equals_numpy_float32(kernels, chunking):
    k32, _ = kernels
    src = _narrow_values()
    n = len(src)
    if chunking == "one":
        chunks = [0, n]
    elif chunking == "split_matrices":   # chunk boundaries that cut through 8 x 8 blocks at odd offsets
        chunks = [0, 37, 1000, 4097, 65_537, n - 3, n]
    else:                                # many small chunks, then the rest
        chunks = [0, 1, 2, 3, 5, 8, 13, 21, 34, 55, 89, n]
    got, flag = _narrow(k32, src, np.asarray(chunks, dtype=np.int64))
    with np.errstate(over="ignore"):
        want = src.astype(np.float32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))   # bitwise, -0.0 and subnormals included
    assert flag == 0                                                    # Inf inputs stay Inf without a flag


def test_narrowing_flags_entries_above_the_float_range(kernels):
    k32, _ = kernels
    f32max = float(np.finfo(np.float32).max)
    for big in (f32max * (1 + 2.0 ** -23), 3.5e38, -1e39, 1e300):
        src = np.concatenate([np.ones(1000), [big], np.ones(77)])
        got, flag = _narrow(k32, src, np.asarray([0, 500, len(src)], dtype=np.int64))
        assert flag == 1 and np.isinf(got[1000]) and np.all(got[:1000] == 1.0)


# ---------------------------------------------------------------------------------------------------------------
# end to end on one GPU: a Double and a Single handle on the same matrix
# ---------------------------------------------------------------------------------------------------------------
def _config(name):
    from hymls_b200 import driver
    p = driver.parse_parameter_list(open(os.path.join(ROOT, "configs", name)).read())
    p.pop("Driver", None)
    return p


def _const_pressure(n, dof):
    V = np.zeros((n, 1))
    V[dof - 1::dof, 0] = 1.0
    return V / np.linalg.norm(V)


def _case(name):
    """(params dict, A, border V or None)"""
    from tests.common import make_params
    from tests.conftest import load_fixture
    from tests.test_gpu_parity import dictify
    gmres = {"Krylov Method": "GMRES", "Initial Vector": "Zero", "Left or Right Preconditioning": "Right",
             "Iterative Solver": {"Maximum Iterations": 300, "Num Blocks": 300, "Convergence Tolerance": 1e-8}}
    if name == "laplace128":
        return _config("laplace.xml"), sp.csr_matrix(hb.galeri.create_matrix("Laplace", 2, 128)), None
    if name == "stokes2d128":
        return _config("stokes2D.xml"), sp.csr_matrix(-hb.galeri.create_matrix("Stokes-C", 2, 128)), None
    if name == "skew16":
        A, _, _ = load_fixture("cavity3d_16_Re0")
        p = dictify(make_params("Stokes-C", 3, 16, 4, 2, 2, Partitioner="Skew Cartesian"))
        p["Solver"] = gmres
        return p, A, None
    assert name == "bordered64"
    A, _, _ = load_fixture("cavity2d_64_Re0")
    p = dictify(make_params("Stokes-C", 2, 64, 4, 2, Fix_Pressure_Level=False))
    p["Solver"] = gmres
    return p, A, _const_pressure(A.shape[0], 3)


def _build(p, A, V, precision):
    import copy
    q = copy.deepcopy(p)
    q["Preconditioner"]["Subdomain Inverse Precision"] = precision
    P = hb.Preconditioner(A, q, hb.galeri.create_testvector(A))
    P.Initialize()
    if V is not None:
        P.SetBorder(V)
    P.Compute()
    return P


def _rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


CASES = ["laplace128", "stokes2d128", "skew16", "bordered64"]


@pytest.fixture(scope="module", params=CASES)
def pair(request):
    p, A, V = _case(request.param)
    return request.param, p, A, V, _build(p, A, V, "Double"), _build(p, A, V, "Single")


def test_single_store_is_float32_of_double(pair):
    name, _, _, _, D, S = pair
    for lev in range(D.NumLevels()):
        a64, a32 = D.DebugArray("a11inv", lev), S.DebugArray("a11inv", lev)
        assert len(a32) == len(a64) > 0
        assert np.array_equal(a32, a64.astype(np.float32).astype(np.float64))
        assert not np.array_equal(a32, a64)
        for arr in ("blkinv", "redval"):
            assert np.array_equal(S.DebugArray(arr, lev), D.DebugArray(arr, lev)), (name, arr, lev)
    last = D.NumLevels() - 1
    assert np.array_equal(S.DebugArray("coarseinv", last), D.DebugArray("coarseinv", last))


def test_single_apply_inverse_is_close_to_double(pair):
    import torch
    name, _, A, V, D, S = pair
    n = A.shape[0]
    rng = np.random.default_rng(3)
    errs = []
    if V is None:
        for nvec in (1, 3):
            B = rng.uniform(-1, 1, (n, nvec)) if nvec > 1 else rng.uniform(-1, 1, n)
            xd, xs = D.ApplyInverse(B), S.ApplyInverse(B)
            errs.append(_rel(xs, xd))
            assert errs[-1] <= SINGLE_TOL and not np.array_equal(xs, xd)
            assert np.array_equal(S.ApplyInverse(B), xs)                        # a fixed operator: bitwise repeatable
            Bt = torch.from_numpy(np.ascontiguousarray(B.T)).cuda()            # device buffers, (nvec, n)
            xdd, xsd = D.ApplyInverse(Bt).cpu().numpy(), S.ApplyInverse(Bt).cpu().numpy()
            errs.append(_rel(xsd, xdd))
            assert errs[-1] <= SINGLE_TOL and not np.array_equal(xsd, xdd)
            assert np.array_equal(S.ApplyInverse(Bt).cpu().numpy(), xsd)
    else:
        B, T = rng.uniform(-1, 1, n), rng.uniform(-1, 1, V.shape[1])
        Xd, Sd = D.ApplyInverseBordered(B, T)
        Xs, Ss = S.ApplyInverseBordered(B, T)
        errs += [_rel(Xs, Xd), _rel(Ss, Sd)]
        assert max(errs) <= SINGLE_TOL and not np.array_equal(Xs, Xd)
        Xs2, Ss2 = S.ApplyInverseBordered(B, T)
        assert np.array_equal(Xs2, Xs) and np.array_equal(Ss2, Ss)
    print("%s: Single vs Double ApplyInverse rel diff %s" % (name, ", ".join("%.2e" % e for e in errs)))


def test_single_krylov_converges_like_double(pair):
    name, p, A, V, D, S = pair
    b = A @ np.random.default_rng(4).uniform(-1, 1, A.shape[0])
    # Both precisions solve to 1e-8 (laplace.xml and stokes2D.xml ask for 1e-10).  The solver stops on its recurrence
    # residual; the explicit residual ||b - A x|| / ||b|| of the returned x is 1.0 .. 1.4 times that for Double as
    # well (measured on a B200: 1.13e-8 for laplace128, 1.03e-8 for stokes2d128, 1.36e-8 for the 128^3 bench
    # problem), so both are held to 2 tol.
    tol = 1e-8
    its = {}
    for key, P in (("Double", D), ("Single", S)):
        sol = hb.Solver(P)
        sol.SetTolerance(tol)
        sol.ApplyInverse(b)
        assert sol.info["converged"] and sol.info["explicit_rel_residual"] <= 2 * tol, (name, key, sol.info)
        its[key] = sol.num_iter
    print("%s: %s %d its, Single %d its" % (name, p["Solver"]["Krylov Method"], its["Double"], its["Single"]))
    assert abs(its["Single"] - its["Double"]) <= 1


def test_single_recompute_equals_a_fresh_handle(pair):
    name, p, A, V, D, S = pair
    if V is not None:
        pytest.skip("the recompute path is checked on the unbordered cases")
    A2 = A.copy()
    A2.data = A.data * (1.0 + 1e-3 * np.random.default_rng(6).uniform(-1, 1, A.nnz))
    S.SetMatrix(A2)
    S.Compute()
    F = _build(p, A2, None, "Single")
    b = np.random.default_rng(7).uniform(-1, 1, A.shape[0])
    assert np.array_equal(S.ApplyInverse(b), F.ApplyInverse(b))
    assert np.array_equal(S.DebugArray("a11inv", 0), F.DebugArray("a11inv", 0))
    S.SetMatrix(A)                       # leave the module's handle as it was built
    S.Compute()


def test_single_stats(pair):
    _, _, _, _, D, S = pair
    sd, ss = D.Stats(), S.Stats()
    assert sd["a11_entry_bytes"] == 8 and ss["a11_entry_bytes"] == 4
    assert ss["bytes_a11_level0"] == sd["bytes_a11_level0"] / 2 > 0


# ---------------------------------------------------------------------------------------------------------------
# owner-distributed path: Single on N ranks against Single on one GPU (the FP64 inverses do not depend on the rank
# count, so neither do the narrowed ones); the tolerances of test_gpu_bordered_dist.py
# ---------------------------------------------------------------------------------------------------------------
def _worker(rank, world, port, out):
    import torch
    import torch.distributed as dist
    from tests.test_gpu_bordered_dist import TOL_S, TOL_X, _case as bcase
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

        solver = {"Krylov Method": "GMRES", "Initial Vector": "Zero", "Left or Right Preconditioning": "Right",
                  "Iterative Solver": {"Maximum Iterations": 300, "Num Blocks": 300, "Convergence Tolerance": 1e-8}}
        for name in ("m2-general", "cube32-skew"):
            p, A, V, W, Cm, b = bcase(name)
            pd = _dictify(p)
            pd["Solver"] = solver
            pd["Preconditioner"]["Subdomain Inverse Precision"] = "Single"
            P = hb.Preconditioner(A, pd, hb.galeri.create_testvector(A))
            P.CommInit(comm_id(), rank, world)
            P.Initialize()
            P.Compute()
            Q = hb.Preconditioner(A, pd, hb.galeri.create_testvector(A))
            Q.Initialize()
            Q.Compute()
            rows = P.OwnedRows()
            rng = np.random.default_rng(2)
            B = rng.uniform(-1, 1, A.shape[0])
            x1 = Q.ApplyInverse(B)
            x = P.ApplyInverseDist(B[rows].copy())
            num = allsum([np.sum((x - x1[rows]) ** 2), np.sum(x1[rows] ** 2)])
            r = {"x_rel": float(np.sqrt(num[0] / num[1]))}
            sp_, sq = hb.Solver(P), hb.Solver(Q)
            sp_.ApplyInverse(b)
            sq.ApplyInverse(b)
            r["its"], r["its_single_gpu"] = sp_.num_iter, sq.num_iter
            r["converged"] = [bool(sp_.info["converged"]), bool(sq.info["converged"])]
            T = rng.uniform(-1, 1, V.shape[1])
            for H in (P, Q):
                H.SetBorder(V, W, Cm)
                H.Compute()
            X1, S1 = Q.ApplyInverseBordered(B, T)
            xb, Sb = P.ApplyInverseBorderedDist(B[rows].copy(), T.copy())
            num = allsum([np.sum((xb - X1[rows, 0]) ** 2), np.sum(X1[rows, 0] ** 2)])
            r["xb_rel"] = float(np.sqrt(num[0] / num[1]))
            r["sb_rel"] = float(np.linalg.norm(Sb - S1[:, 0]) / np.linalg.norm(S1[:, 0]))
            sp_, sq = hb.Solver(P), hb.Solver(Q)
            sp_.ApplyInverse(b)
            sq.ApplyInverse(b)
            r["its_b"], r["its_b_single_gpu"] = sp_.num_iter, sq.num_iter
            r["tol_x"], r["tol_s"] = TOL_X, TOL_S
            res[name] = r
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


def _dictify(p):
    return {k: (_dictify(v) if isinstance(v, dict) else v) for k, v in p.items()}


@pytest.mark.parametrize("world", [2, 4])
def test_single_on_the_owner_path_matches_one_gpu(world):
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
    for name, r in res.items():
        print("%s on %d ranks: %s" % (name, world, r))
        assert r["x_rel"] <= r["tol_x"] and r["xb_rel"] <= r["tol_x"] and r["sb_rel"] <= r["tol_s"]
        assert r["converged"][0] == r["converged"][1]
        assert r["its"] == r["its_single_gpu"] and r["its_b"] == r["its_b_single_gpu"]
