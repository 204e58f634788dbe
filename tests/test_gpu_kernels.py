"""The CUDA kernels one launcher at a time, on shapes chosen on purpose.

The parity tests run the whole preconditioner, so which kernel path runs depends on the block sizes the
partitioner happens to produce, and a kernel that is wrong in one rare case can hide behind the rest of the
pipeline.  Here tests/kernel_harness.cpp exposes the launchers of libhymls_b200.so (hymls_b200/csrc/kernels.hpp)
as extern "C" functions, and every test calls one of them on torch-owned device memory and compares the result with
a reference of the same operation:

* EXACT: inputs are small integers (|a| <= 2^8, at most a few thousand terms per sum), so FP64 computes every
  product and every partial sum exactly, in any order.  The kernel's result must be bitwise equal to numpy's;
  any index, offset or masking error fails whatever its size.  Used for denseGemm, the GEMV family, spmv and
  multiAxpy.
* EXTENDED: longdouble (oracle/extended.py: LAPACK LU + iterative refinement with extended-precision residuals,
  or math.fsum), with a tolerance derived from the rounding-error bound of the operation.  Used for the
  inversions, the Newton-Schulz steps, multiDot and the Householder transforms.  Inverses too large for the
  longdouble reference are checked through their normwise residual, computed with FP64 torch on the GPU.

u = 2^-53 is the unit roundoff and gamma(k) = k u / (1 - k u) the factor of Higham's bound for a k-term sum
(Accuracy and Stability of Numerical Algorithms, 2nd ed., section 3.1); it holds for every summation order, so
also for the tree and tensor-core orders of the kernels.
"""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest
import scipy.linalg as sla
import scipy.sparse as sp

from oracle import extended as ox

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_DIR = os.path.join(ROOT, "hymls_b200")
LD = np.longdouble
U = 2.0 ** -53
EPS = 2.0 ** -52


def gamma(k):
    return k * U / (1.0 - k * U)


# ---------------------------------------------------------------------------------------------------------------
# the harness
# ---------------------------------------------------------------------------------------------------------------
_vp, _i32, _i64, _dbl = C.c_void_p, C.c_int, C.c_int64, C.c_double
_GEMV = [_vp] * 16 + [_i32, _i32]  # GemvArgs, flat, in the order of the struct
_TAIL = [_vp, C.POINTER(C.c_int64)]  # stream, launch counter
WRAPPERS = {
    "kh_invert_batched": [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp] + _TAIL,
    "kh_refine_inverse_batched": [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32] + _TAIL,
    "kh_refine_inverse_sparse": [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32] + _TAIL,
    "kh_dense_gemm": [_vp, _i32, _vp, _i32, _vp, _i32, _i32, _i32, _i32, _dbl, _dbl] + _TAIL,
    "kh_batched_gemv": _GEMV + [_i32, _i32] + _TAIL,
    "kh_batched_gemv_multi": _GEMV + [_i32, _i32, _i32, _i64, _i64, _i64, _vp] + _TAIL,
    "kh_small_gemv": _GEMV + [_vp, _i32, _i32, _vp] + _TAIL,
    "kh_cta_gemv": _GEMV + [_vp, _i32, _i32] + _TAIL,
    "kh_multi_dot": [_vp, _i64, _i32, _vp, _i64, _vp, _vp, _i32, _vp] + _TAIL,
    "kh_multi_axpy": [_vp, _i64, _i32, _vp, _vp, _i64, _dbl] + _TAIL,
    "kh_spmv": [_vp, _vp, _vp, _vp, _vp, _i64, _dbl, _vp, _vp, _dbl] + _TAIL,
    "kh_householder": [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp] + _TAIL,
    "kh_gemv_rows_per_item": [],
    "kh_multi_dot_blocks": [],
}


def _build_harness(outdir):
    cuda = os.environ.get("CUDA_HOME") or "/usr/local/cuda"
    so = os.path.join(str(outdir), "kernel_harness.so")
    cmd = ["/usr/bin/g++", "-std=c++17", "-Wall", "-Werror", "-fPIC", "-shared",
           "-I" + os.path.join(LIB_DIR, "csrc"), "-I" + os.path.join(cuda, "include"),
           os.path.join(ROOT, "tests", "kernel_harness.cpp"),
           "-L" + LIB_DIR, "-lhymls_b200", "-L" + os.path.join(cuda, "lib64"), "-lcudart",
           "-Wl,-rpath," + LIB_DIR, "-Wl,-rpath," + os.path.join(cuda, "lib64"), "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = C.CDLL(so)
    for name, argtypes in WRAPPERS.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    return lib


@pytest.fixture(scope="module")
def harness_lib(tmp_path_factory):
    return _build_harness(tmp_path_factory.mktemp("kernel_harness"))


def test_harness_compiles_links_and_resolves_every_wrapper(harness_lib):
    # catches drift between kernels.hpp and the launchers the library exports without a GPU
    for name in WRAPPERS:
        assert getattr(harness_lib, name) is not None
    assert harness_lib.kh_gemv_rows_per_item() == 32
    assert harness_lib.kh_multi_dot_blocks() == 592


class Kernels:
    """Calls a wrapper on torch's current stream; returns the number of kernel launches it reported.

    Device arguments are given as torch tensors (or numpy arrays, copied to the device here) and passed as their
    data pointers; this call holds a reference to each of them until the kernels have finished, so no buffer
    can be freed and reused while a kernel reads it."""

    def __init__(self, lib):
        import torch
        self.lib, self.torch = lib, torch

    def __call__(self, name, *args):
        held = [_d(a) if isinstance(a, np.ndarray) else a for a in args]
        raw = [a.data_ptr() if isinstance(a, self.torch.Tensor) else a for a in held]
        launches = C.c_int64(0)
        stream = self.torch.cuda.current_stream().cuda_stream
        rc = getattr(self.lib, name)(*raw, stream, C.byref(launches))
        assert rc == 0, "%s returned %d" % (name, rc)
        del held
        return launches.value


@pytest.fixture(scope="module")
def kh(harness_lib):
    return Kernels(harness_lib)


def _d(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda")


def _h(t):
    return t.cpu().numpy()


# ---------------------------------------------------------------------------------------------------------------
# batched inversion (gj.cu)
# ---------------------------------------------------------------------------------------------------------------
# invertBatched picks the panel kernel per matrix and panel by the active rows R = np - k0 of the 32-column panel
# starting at k0: k_gj_panel_full for R <= 824, k_gj_panel_smem<8> up to 3072, k_gj_panel_smem<4> up to 6144,
# k_gj_panel beyond.  The host launches k_gj_panel_full for every panel of the batch and each taller-panel kernel
# for every panel whose largest active part npMax - k0 exceeds the kernel's lower limit, so
#   launches = 1 (k_pad_identity) + panels * 3 (k_gj_panel_full, k_gj_swaplist, k_gj_update)
#              + #panels(R > 824) + #panels(R > 3072) + #panels(R > 6144) + 2 (k_gj_perm, k_gj_gather),
# panels = ceil(npMax / 32).  The table gives those numbers for each npMax used below.
GJ_LAUNCHES = {16: 6, 40: 9, 200: 24,
               824: 81,     # 26 panels, none taller than 824 rows
               832: 82,     # + 1 k_gj_panel_smem<8> (k0 = 0)
               3072: 362,   # 96 panels, 71 of them taller than 824
               3080: 366,   # 97 panels, 71 > 824, 1 k_gj_panel_smem<4> (k0 = 0)
               6144: 842,   # 192 panels, 167 > 824, 96 > 3072
               6152: 847,   # 193 panels, 167 > 824, 97 > 3072, 1 k_gj_panel (k0 = 0)
               6200: 853}   # 194 panels, 168 > 824, 98 > 3072, 2 k_gj_panel (k0 = 0, 32: rows above the panel)


def _pack(mats, nps):
    """Row-major np x np blocks, zero padding (the launcher puts the identity on the padding diagonal)."""
    off = np.zeros(len(nps) + 1, dtype=np.int64)
    off[1:] = np.cumsum(np.asarray(nps, dtype=np.int64) ** 2)
    W = np.zeros(int(off[-1]))
    for m, (A, q) in enumerate(zip(mats, nps)):
        blk = np.zeros((q, q))
        blk[:A.shape[0], :A.shape[0]] = A
        W[off[m]:off[m + 1]] = blk.ravel()
    return W, off


def _blocks(flat, off, nps):
    return [flat[off[m]:off[m + 1]].reshape(q, q) for m, q in enumerate(nps)]


def invert(kh, mats, nps):
    """invertBatched on a batch: (padded inverses on the device, offsets, info, launches, pivots)."""
    import torch
    count, npmax = len(mats), max(nps)
    W, off = _pack(mats, nps)
    dW = _d(W)
    dF = torch.full_like(dW, float("nan"))  # every entry of F must be written
    dOff, dN = _d(off[:-1]), _d(np.asarray([A.shape[0] for A in mats], dtype=np.int32))
    dNp = _d(np.asarray(nps, dtype=np.int32))
    piv = torch.full((count * npmax,), -1, dtype=torch.int32, device="cuda")
    perm = torch.empty(count * npmax, dtype=torch.int32, device="cuda")
    swap = torch.empty(count * 128, dtype=torch.int32, device="cuda")
    info = torch.zeros(1, dtype=torch.int32, device="cuda")
    launches = kh("kh_invert_batched", dW, dF, dOff, dN, dNp, count, npmax, piv, perm,
                  swap, info)
    del dW
    return dF, off, int(info.item()), launches, _h(piv).reshape(count, npmax)


def _ext_inverse(A):
    """Extended-precision inverse (longdouble iterative refinement of LAPACK's LU solve)."""
    return ox._RefinedDenseLU(A).solve(np.eye(A.shape[0]))


def _forward_error(X, A):
    """||X - inv(A)||_F / ||inv(A)||_F against the extended reference, and its tolerance 8 n u kappa_2(A).

    Gauss-Jordan elimination with partial pivoting is forward stable: its error is bounded like that of an
    LU-based inverse, c n u kappa(A) times the growth of the factors (Higham, Accuracy and Stability, section
    14.4), and the growth is small for these matrices.  c = 8 leaves room for the constant and for the mix of
    norms (LAPACK's inverses of the 16384 small matrices below reach half of the bound with c = 2)."""
    Xe = _ext_inverse(A)
    err = float(np.linalg.norm((X.astype(LD) - Xe).astype(np.float64)) / np.linalg.norm(Xe.astype(np.float64)))
    n = A.shape[0]
    return err, _fe_tol(A, n)


def _fe_tol(A, n):
    return 8 * n * U * np.linalg.cond(A)


def _residual(A, X):
    """Normwise residual ||I - A X||_F / (||A||_F ||X||_F), FP64 on the GPU.  A stable inverse has c_n u; the
    GEMM that forms it adds at most gamma(n) (Frobenius norms), so n eps bounds both."""
    import torch
    dA = _d(A)
    dX = X if isinstance(X, torch.Tensor) else _d(X)
    R = torch.eye(A.shape[0], dtype=torch.float64, device="cuda") - dA @ dX
    return float(torch.linalg.norm(R) / (torch.linalg.norm(dA) * torch.linalg.norm(dX)))


def _check_padding(F, n):
    q = F.shape[0]
    assert np.array_equal(F[n:, n:], np.eye(q - n)), "padding block of the inverse is not the identity"
    assert not F[:n, n:].any() and not F[n:, :n].any(), "padding rows / columns of the inverse are not zero"


def _gaussian(n, rng):
    return rng.standard_normal((n, n))


def _saddle(n, rng, scale=1.0):
    """[[s K, s B], [B^T, 0]]: the zero block forces pivot rows from below the panel; s = nx^2 scales the
    velocity rows against the pressure rows as in the Stokes blocks."""
    n2 = n // 3
    n1 = n - n2
    G = rng.standard_normal((n1, n1))
    K = G @ G.T / n1 + np.eye(n1)
    B = rng.standard_normal((n1, n2))
    A = np.zeros((n, n))
    A[:n1, :n1], A[:n1, n1:], A[n1:, :n1] = scale * K, scale * B, B.T
    return A


def _stokes_scaled(n, rng):
    return _saddle(n, rng, scale=32.0 ** 2)


def _permuted_dominant(n, rng):
    """Rows of a column diagonally dominant D, permuted so that partial pivoting meets an interchange with the same
    outside row several times in one panel.  For such a D every Schur complement is column diagonally dominant too,
    so the pivot of column c is the row that currently holds D's row c.  A chain (p; c1 < c2 < ... < cL) puts
    D[c1] in row p, D[c(i+1)] in row c(i) and D[p] in row cL: column c1 swaps rows c1 and p, after which p holds
    D[c2], so column c2 pivots on row p again, and so on -- L interchanges with row p."""
    D = rng.uniform(-1.0, 1.0, (n, n))
    D[np.arange(n), np.arange(n)] = n * np.where(rng.random(n) < 0.5, -1.0, 1.0)
    sigma = np.arange(n)  # row i of A is row sigma[i] of D
    chains = [(n // 2, [0, 1, 2, 3]),                  # four times in a row, panel 0
              (n - 3, [5, 7, 9, 11]), ((2 * n) // 3, [6, 8, 10]),  # two outside rows interleaved
              (31, [12, 20, 25]),                     # a chain inside the panel
              ((n // 2) + 1, [28, 30, 33, 40])]       # an outside row hit in panel 0 and again in panel 1
    for p, cols in chains:
        sigma[p] = cols[0]
        for a, b in zip(cols[:-1], cols[1:]):
            sigma[a] = b
        sigma[cols[-1]] = p
    assert np.array_equal(np.sort(sigma), np.arange(n))
    return D[sigma]


FAMILIES = {"gaussian": _gaussian, "saddle": _saddle, "stokes_scaled": _stokes_scaled,
            "permuted_dominant": _permuted_dominant}
EXT_MAX = 520  # largest n checked against the longdouble reference (its cost grows like n^3 in longdouble)


def _check_inverse(F, A, what):
    """Forward error (n <= EXT_MAX) or normwise residual next to LAPACK's; returns the measured numbers."""
    n = A.shape[0]
    X = F[:n, :n]
    if n <= EXT_MAX:
        err, tol = _forward_error(X, A)
        assert err <= tol, "%s: forward error %.3e > %.3e" % (what, err, tol)
        return {"forward_error": err, "tol": tol}
    res = _residual(A, X)
    res_lapack = _residual(A, sla.inv(A))
    tol = n * EPS
    assert res <= tol, "%s: residual %.3e > %.3e (LAPACK %.3e)" % (what, res, tol, res_lapack)
    return {"residual": res, "residual_lapack": res_lapack, "tol": tol}


def _report(what, numbers):
    print("[gpu_kernels] %s %s" % (what, " ".join("%s=%.3e" % kv for kv in numbers.items())))


@pytest.mark.gpu
@pytest.mark.parametrize("npad,n", [(824, 824), (832, 827), (3072, 3072), (3080, 3075), (6144, 6144), (6152, 6147),
                                    (6200, 6200)])
def test_invert_single_matrix_at_panel_kernel_boundaries(kh, npad, n):
    """Both sides of each panel-kernel limit; np = 6200 also gives k_gj_panel a panel with rows above it (at
    np = 6152 it only factors the first panel).  Reference: normwise residual next to LAPACK's (n > EXT_MAX)."""
    rng = np.random.default_rng(npad)
    A = _gaussian(n, rng)
    dF, off, info, launches, piv = invert(kh, [A], [npad])
    assert info == 0
    assert launches == GJ_LAUNCHES[npad]
    F = _h(dF)
    _check_padding(F.reshape(npad, npad), n)
    _report("boundary np=%d n=%d" % (npad, n), _check_inverse(F.reshape(npad, npad), A, "np=%d" % npad))


@pytest.mark.gpu
@pytest.mark.parametrize("family", sorted(FAMILIES))
@pytest.mark.parametrize("npad", [200, 832, 3080, 6152])  # first panel in each of the four panel kernels
def test_invert_matrix_families(kh, family, npad):
    """Reference: extended forward error (np = 200) or normwise residual next to LAPACK's."""
    rng = np.random.default_rng([npad, len(family)])
    n = npad - 5
    A = FAMILIES[family](n, rng)
    dF, off, info, launches, piv = invert(kh, [A], [npad])
    assert info == 0 and launches == GJ_LAUNCHES[npad]
    F = _h(dF).reshape(npad, npad)
    _check_padding(F, n)
    if family == "permuted_dominant":
        # the construction does what it claims: LAPACK and the kernel pick the same (unambiguous) pivots, and
        # row n/2 is the pivot of the four first columns
        assert np.array_equal(piv[0, :n], sla.lu_factor(A)[1])
        assert np.array_equal(piv[0, n:], np.arange(n, npad))
        assert np.array_equal(piv[0, :4], [n // 2] * 4)
    _report("family %s np=%d n=%d" % (family, npad, n), _check_inverse(F, A, family))


@pytest.mark.gpu
def test_invert_mixed_batch_moves_between_bands_and_is_reproducible(kh):
    """np = 8, 40 (extended forward error) and 824, 832, 3080 (normwise residual) in one batch: at k0 = 0 the
    matrices use three different panel kernels, and 832 / 3080 move to the lower bands as k0 grows."""
    rng = np.random.default_rng(7)
    nps = [8, 40, 824, 832, 3080]
    ns = [8, 35, 824, 827, 3080]
    mats = [_gaussian(n, rng) for n in ns]
    dF, off, info, launches, piv = invert(kh, mats, nps)
    assert info == 0 and launches == GJ_LAUNCHES[3080]
    F = _h(dF)
    for m, (A, q) in enumerate(zip(mats, nps)):
        Fm = _blocks(F, off, nps)[m]
        _check_padding(Fm, A.shape[0])
        _report("mixed np=%d n=%d" % (q, A.shape[0]), _check_inverse(Fm, A, "mixed batch np=%d" % q))
    dF2, _, _, _, piv2 = invert(kh, mats, nps)
    assert np.array_equal(_h(dF2), F) and np.array_equal(piv2, piv), "two inversions of one batch differ"


@pytest.mark.gpu
def test_invert_batch_of_16384_small_matrices(kh):
    """Callers chunk at 16384 matrices; k_gj_update puts the matrix on grid.y.  Reference: LAPACK's inverses
    refined by one Newton-Schulz step in longdouble (error ~ (kappa eps)^2), forward error per matrix."""
    rng = np.random.default_rng(16384)
    count = 16384
    nps = rng.choice([8, 16], count).tolist()
    ns = [int(rng.integers(1, q + 1)) for q in nps]
    mats = [_gaussian(n, rng) + n * np.eye(n) * (m % 2) for m, n in enumerate(ns)]
    dF, off, info, launches, _ = invert(kh, mats, nps)
    assert info == 0 and launches == GJ_LAUNCHES[16]
    F = _blocks(_h(dF), off, nps)
    worst = 0.0
    for n in sorted(set(ns)):
        idx = [m for m in range(count) if ns[m] == n]
        A = np.stack([mats[m] for m in idx])
        X = np.stack([F[m][:n, :n] for m in idx])
        Xl = np.linalg.inv(A).astype(LD)
        Al = A.astype(LD)
        Xe = Xl + Xl @ (np.eye(n, dtype=LD) - Al @ Xl)
        err = (np.linalg.norm((X - Xe).astype(np.float64), axis=(1, 2))
               / np.linalg.norm(Xe.astype(np.float64), axis=(1, 2)))
        tol = _fe_tol(A, n)
        bad = np.nonzero(~(err <= tol))[0]
        assert bad.size == 0, "n=%d: matrices %s, errors %s > %s" % (n, [idx[b] for b in bad[:5]], err[bad[:5]],
                                                                     tol[bad[:5]])
        worst = max(worst, float((err / tol).max()))
        for m in idx[:50]:
            _check_padding(F[m], n)
    _report("batch16384", {"worst_error_over_tol": worst})


# one matrix per panel kernel: np = 40 -> k_gj_panel_full, 832 -> k_gj_panel_smem<8>, 3080 -> k_gj_panel_smem<4>,
# 6152 -> k_gj_panel (column 3 lies in the panel k0 = 0)
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["zero_column", "nan_column"])
@pytest.mark.parametrize("npad", [40, 832, 3080, 6152])
def test_invert_flags_singular_matrix_and_keeps_the_others(kh, kind, npad):
    """An exactly zero (or all-NaN) column gives a pivot that is not > 0: info = index + 1.  The bad matrix turns
    into NaN / Inf values, which stay inside its own block.  Reference for the others: extended forward error."""
    rng = np.random.default_rng([npad, len(kind)])
    bad = _gaussian(npad, rng)
    bad[:, 3] = 0.0 if kind == "zero_column" else np.nan
    good = [_gaussian(40, rng), _gaussian(33, rng)]
    dF, off, info, launches, _ = invert(kh, [good[0], bad, good[1]], [40, npad, 40])
    assert info == 2
    assert launches == GJ_LAUNCHES[npad]
    F = _blocks(_h(dF), off, [40, npad, 40])
    for m, A in ((0, good[0]), (2, good[1])):
        _check_padding(F[m], A.shape[0])
        _check_inverse(F[m], A, "healthy matrix %d next to a singular one" % m)


# ---------------------------------------------------------------------------------------------------------------
# Newton-Schulz refinement X1 = X0 + X0 (I - A X0)
# ---------------------------------------------------------------------------------------------------------------
REFINE_NPS = [8, 40, 72, 200, 520]
REFINE_NS = [8, 35, 72, 193, 515]


def _refine_inputs(rng):
    """Padded originals A (identity in the padding, as the kernels use them) and perturbed inverses X0 with
    ||I - A X0|| ~ 1e-6, so that one step has a residual to square."""
    mats = [_gaussian(n, rng) + 2.0 * math.sqrt(n) * np.eye(n) for n in REFINE_NS]
    Ap, X0 = [], []
    for A, q in zip(mats, REFINE_NPS):
        n = A.shape[0]
        a = np.eye(q)
        a[:n, :n] = A
        x = np.eye(q)
        x[:n, :n] = np.linalg.inv(A) * (1.0 + 1e-6 * rng.standard_normal((n, n)))
        Ap.append(a)
        X0.append(x)
    return mats, Ap, X0


def _check_newton_schulz(X1, A, X0, what):
    """X1 against the exact step in longdouble.  Rounding of the FP64 step (Frobenius norms, N = np):
         R^ = I - A X0 + E1,  ||E1|| <= gamma(N+1) ||A|| ||X0||       (the sparse residual sums fewer terms)
         T^ = X0 R^ + E2,     ||E2|| <= gamma(N) ||X0|| ||R^||
         X1^ = fl(X0 + T^),   ||E3|| <= u ||X1^||
       so ||X1^ - X1|| <= ||X0|| ||E1|| + ||E2|| + ||E3||.  Also I - A X1 = (I - A X0)^2 exactly, so the residual
       must drop to about its square: ||I - A X1^|| <= ||I - A X0||^2 + ||A|| * (that bound)."""
    N = A.shape[0]
    Al, X0l = A.astype(LD), X0.astype(LD)
    I = np.eye(N, dtype=LD)
    R0 = I - Al @ X0l
    X1e = X0l + X0l @ R0
    nA, nX0, nR0 = (float(np.linalg.norm(M.astype(np.float64))) for M in (A, X0, R0))
    bound = nX0 * gamma(N + 1) * nA * nX0 + gamma(N) * nX0 * (nR0 + gamma(N + 1) * nA * nX0) \
        + U * float(np.linalg.norm(X1))
    err = float(np.linalg.norm((X1.astype(LD) - X1e).astype(np.float64)))
    assert err <= bound, "%s: ||X1 - X1_exact|| = %.3e > %.3e" % (what, err, bound)
    res1 = float(np.linalg.norm((I - Al @ X1.astype(LD)).astype(np.float64)))
    assert res1 <= nR0 ** 2 + nA * bound, "%s: residual %.3e after the step, %.3e before" % (what, res1, nR0)
    return {"step_error": err, "step_bound": bound, "residual_before": nR0, "residual_after": res1}


@pytest.mark.gpu
def test_refine_inverse_batched_squares_the_residual(kh):
    """Reference: the exact Newton-Schulz step in longdouble, with the FP64 rounding bound."""
    import torch
    rng = np.random.default_rng(11)
    mats, Ap, X0 = _refine_inputs(rng)
    A_flat, off = _pack(mats, REFINE_NPS)  # originals without the padding identity: the launcher adds it
    X_flat, _ = _pack(X0, REFINE_NPS)
    dA, dF = _d(A_flat), _d(X_flat)
    dR = torch.full_like(dA, float("nan"))
    count, npmax = len(mats), max(REFINE_NPS)
    launches = kh("kh_refine_inverse_batched", dA, dF, dR, off[:-1],
                  np.asarray(REFINE_NS, dtype=np.int32), np.asarray(REFINE_NPS, dtype=np.int32),
                  count, npmax)
    assert launches == 4  # k_pad_identity, two k_refine_gemm, k_refine_add
    X1 = _blocks(_h(dF), off, REFINE_NPS)
    for m, q in enumerate(REFINE_NPS):
        _report("refine_batched np=%d" % q, _check_newton_schulz(X1[m], Ap[m], X0[m], "np=%d" % q))


def _dense_fill_list(sparse_mats, off, dst_base, lead, rng):
    """The dense-fill list of the sparse originals, as buildA11List makes it: value index into one value array,
    absolute dense position dstBase + off[m] + r np + c, ascending per matrix; `lead` unrelated entries first so
    that listPtr does not start at 0."""
    vals, src, dst, ptr = [], [], [], [lead]
    pos = 0
    for m, S in enumerate(sparse_mats):
        q = int(round(math.sqrt(off[m + 1] - off[m])))
        S = sp.csr_matrix(S)
        S.sort_indices()
        rows = np.repeat(np.arange(S.shape[0]), np.diff(S.indptr))
        dst.append(dst_base + off[m] + rows.astype(np.int64) * q + S.indices)
        vals.append(S.data)
        src.append(np.arange(pos, pos + S.nnz, dtype=np.int64))
        pos += S.nnz
        ptr.append(ptr[-1] + S.nnz)
    val = np.concatenate(vals)
    # the values sit in a shuffled array: src is a real indirection
    shuffle = rng.permutation(val.size)
    val_shuffled = np.empty_like(val)
    val_shuffled[shuffle] = val
    src = shuffle[np.concatenate(src)]
    junk = np.zeros(lead, dtype=np.int64)
    return (val_shuffled, np.concatenate([junk, src]).astype(np.int64), np.concatenate([junk] + dst).astype(np.int64),
            np.asarray(ptr, dtype=np.int64))


@pytest.mark.gpu
def test_refine_inverse_sparse_squares_the_residual(kh):
    """Residual from the dense-fill list of scipy CSR originals, with a non-zero dstBase and listPtr offset.
    Reference: the exact Newton-Schulz step in longdouble, with the FP64 rounding bound."""
    import torch
    rng = np.random.default_rng(12)
    sparse_mats, Ap, X0 = [], [], []
    for n, q in zip(REFINE_NS, REFINE_NPS):
        S = sp.random(n, n, density=min(1.0, 6.0 / n), random_state=rng, data_rvs=rng.standard_normal, format="csr")
        S = sp.csr_matrix(S + sp.diags(2.0 * math.sqrt(n) * np.ones(n)))
        a = np.eye(q)
        a[:n, :n] = S.toarray()
        x = np.eye(q)
        x[:n, :n] = np.linalg.inv(S.toarray()) * (1.0 + 1e-6 * rng.standard_normal((n, n)))
        sparse_mats.append(S)
        Ap.append(a)
        X0.append(x)
    X_flat, off = _pack(X0, REFINE_NPS)
    dst_base = 1000
    val, src, dst, ptr = _dense_fill_list(sparse_mats, off, dst_base, 7, rng)
    dF = _d(X_flat)
    dT = torch.full_like(dF, float("nan"))
    dR = torch.full_like(dF, float("nan"))
    count, npmax = len(sparse_mats), max(REFINE_NPS)
    launches = kh("kh_refine_inverse_sparse", val, src, dst, ptr, dst_base, dT,
                  dF, dR, off[:-1], np.asarray(REFINE_NS, dtype=np.int32),
                  np.asarray(REFINE_NPS, dtype=np.int32), count, npmax)
    assert launches == 3  # k_refine_residual_sparse, k_refine_gemm, k_refine_add
    X1 = _blocks(_h(dF), off, REFINE_NPS)
    for m, q in enumerate(REFINE_NPS):
        _report("refine_sparse np=%d" % q, _check_newton_schulz(X1[m], Ap[m], X0[m], "np=%d" % q))


# ---------------------------------------------------------------------------------------------------------------
# dense GEMM (gj.cu k_dense_gemm): exact reference
# ---------------------------------------------------------------------------------------------------------------
def _ints(rng, shape, lim=256):
    return rng.integers(-lim, lim + 1, shape).astype(np.float64)


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K", [(8, 40, 200), (40, 200, 8), (200, 8, 40), (200, 200, 200), (34, 66, 98),
                                   (2, 2, 2)])
@pytest.mark.parametrize("alpha,beta", [(1.0, 0.0), (-2.0, 1.0), (0.5, -0.5), (3.0, 0.0)])
def test_dense_gemm_exact(kh, M, N, K, alpha, beta):
    """C = alpha A B + beta C with padded leading dimensions; with beta = 0 C starts as NaN and must not leak.
    Integers: every product and sum is exact, alpha and beta scale exactly -> bitwise equal to numpy."""
    rng = np.random.default_rng([M, N, K])
    lda, ldb, ldc = K + 6, N + 2, N + 10
    A = _ints(rng, (M, lda))
    B = _ints(rng, (K, ldb))
    C0 = np.full((M, ldc), np.nan) if beta == 0.0 else _ints(rng, (M, ldc))
    ref = C0.copy()
    ref[:, :N] = alpha * (A[:, :K] @ B[:, :N]) + (beta * C0[:, :N] if beta != 0.0 else 0.0)
    dC = _d(C0)
    launches = kh("kh_dense_gemm", A, lda, B, ldb, dC, ldc, M, N, K, alpha, beta)
    assert launches == 1
    assert np.array_equal(_h(dC), ref, equal_nan=True)


# ---------------------------------------------------------------------------------------------------------------
# batched GEMV family (apply.cu): exact reference
# ---------------------------------------------------------------------------------------------------------------
# np = 8..72 covers every lane split of k_small_gemv's np <= 64 branch (4/8/16/32 lanes per row, one or two loads)
# and its general branch; 264 / 512 / 520 the CTA and slab kernels; n = np, np - 1, np - 7 ragged padding
GEMV_SHAPES = [(q, n) for q in list(range(8, 73, 8)) + [264, 512, 520] for n in (q, q - 1, q - 7)]
SENTINEL = 0.25  # never a result: the exact results are integers


class GemvCase:
    """A batch of padded matrices (integers everywhere, padding rows and columns included), the GemvArgs inputs
    for a set of options and the exact expected output."""

    def __init__(self, opts, seed, shapes=GEMV_SHAPES, nv=1):
        rng = np.random.default_rng(seed)
        self.opts = set(opts)
        self.shapes = shapes
        self.nv = nv
        self.np_ = np.asarray([q for q, _ in shapes], dtype=np.int32)
        self.n = np.asarray([n for _, n in shapes], dtype=np.int32)
        count = len(shapes)
        self.count = count
        self.matOff = np.zeros(count + 1, dtype=np.int64)
        self.matOff[1:] = np.cumsum(self.np_.astype(np.int64) ** 2)
        self.vecOff = np.zeros(count + 1, dtype=np.int64)
        self.vecOff[1:] = np.cumsum(self.n)
        N = int(self.vecOff[-1])
        self.A = _ints(rng, int(self.matOff[-1]))
        self.mats = [self.A[self.matOff[m]:self.matOff[m + 1]].reshape(q, q) for m, q in enumerate(self.np_)]
        # options
        self.ncols = None
        if "ncols" in opts:  # odd leading column counts; x is zero beyond them
            self.ncols = np.asarray([2 * int(rng.integers(0, (n + 1) // 2)) + 1 for n in self.n], dtype=np.int32)
        self.nrows_lead = None
        if "nrows" in opts:  # leading rows of the first solve (0 and n included)
            lead = [int(rng.integers(0, n + 1)) for n in self.n]
            lead[0], lead[1] = 0, int(self.n[1])
            self.nrows_lead = np.asarray(lead, dtype=np.int32)
        self.rpw = 1 if "rpw1" in opts else 0
        self.mode = 1 if "mode1" in opts else 0
        nin = N + 37 if "gather" in opts else N
        self.gather = rng.permutation(nin)[:N].astype(np.int32) if "gather" in opts else None
        if "outoff" in opts:  # segments in reverse order with gaps
            gaps = rng.integers(0, 5, count)
            outOff, pos = np.zeros(count, dtype=np.int64), 0
            for m in reversed(range(count)):
                pos += int(gaps[m])
                outOff[m] = pos
                pos += int(self.n[m])
            self.outOff, nout = outOff, pos + 3
        else:
            self.outOff, nout = None, N
        nscat = nout + 41 if "scatter" in opts else nout
        self.scatter = rng.permutation(nscat)[:nout].astype(np.int32) if "scatter" in opts else None
        if "same_gather_scatter" in opts:  # ApplyBlockDiagonal gathers and scatters through one index array
            self.scatter = self.gather
            nscat = nin
        self.nin, self.nout = nin, nscat
        # vectors: x_sd (what the kernel must multiply), xsub, xin built from them
        self.xin = np.empty((nv, nin))
        self.xsub = _ints(rng, (nv, N)) if "xsub" in opts else None
        self.xprev = _ints(rng, (nv, N)) if self.mode == 1 else None
        self.xsd = _ints(rng, (nv, N))
        for m in range(count):
            v0, n = self.vecOff[m], self.n[m]
            if self.ncols is not None:
                self.xsd[:, v0 + self.ncols[m]:v0 + n] = 0.0
        for v in range(nv):
            self.xin[v] = _ints(rng, nin)  # entries nobody gathers stay non-zero
            vals = self.xsd[v] + (self.xsub[v] if self.xsub is not None else 0.0)
            if self.gather is not None:
                self.xin[v, self.gather] = vals
            else:
                self.xin[v, :N] = vals

    def dest(self, m, r):
        o = (self.outOff[m] if self.outOff is not None else self.vecOff[m]) + r
        return self.scatter[o] if self.scatter is not None else o

    def expected(self, rows=None):
        """Exact output; rows(m) -> row range computed for matrix m (default all n), untouched: SENTINEL."""
        out = np.full((self.nv, self.nout), SENTINEL)
        for m in range(self.count):
            n, v0 = int(self.n[m]), int(self.vecOff[m])
            r0, r1 = rows(m) if rows else (0, n)
            idx = [self.dest(m, r) for r in range(r0, r1)]
            for v in range(self.nv):
                acc = self.mats[m][r0:r1, :n] @ self.xsd[v, v0:v0 + n]
                out[v, idx] = (self.xprev[v, v0 + r0:v0 + r1] - acc) if self.mode == 1 else acc
        return out

    def owner(self):
        """output position -> (np, n) of the matrix that writes it"""
        own = {}
        for m in range(self.count):
            for r in range(int(self.n[m])):
                own[int(self.dest(m, r))] = self.shapes[m]
        return own

    def items(self, first=None, last=None):
        """(itemMat, itemRow0) as BatchedInverse::setup builds them: slabs of 32 rows (8 rows with rowsPerWarp 1)
        from row first(m) up to row last(m)."""
        rows = 8 * self.rpw if self.rpw else 32
        im, ir = [], []
        for m in range(self.count):
            a = first(m) if first else 0
            b = last(m) if last else int(self.n[m])
            for r0 in range(a, b, rows):
                im.append(m)
                ir.append(r0)
        return np.asarray(im, dtype=np.int32), np.asarray(ir, dtype=np.int32)

    def device(self):
        """Device copies of the inputs and an output buffer full of SENTINEL."""
        d = {"n": _d(self.n), "np": _d(self.np_), "matOff": _d(self.matOff), "vecOff": _d(self.vecOff),
             "A": _d(self.A), "xin": _d(self.xin.ravel())}
        for k in ("outOff", "ncols", "gather", "scatter"):
            a = getattr(self, k)
            d[k] = None if a is None else _d(a)
        d["xsub"] = None if self.xsub is None else _d(self.xsub.ravel())
        d["xprev"] = None if self.xprev is None else _d(self.xprev.ravel())
        d["nrows"] = None if self.nrows_lead is None else _d(self.nrows_lead)
        d["out"] = _d(np.full(self.nv * self.nout, SENTINEL))
        return d

    def gemv_args(self, d, itemMat=None, itemRow0=None, nrows=None):
        return (itemMat, itemRow0, d["n"], d["np"], d["matOff"], d["vecOff"],
                d["outOff"], nrows, d["ncols"], d["A"], d["xin"], d["gather"],
                d["xsub"], d["xprev"], d["out"], d["scatter"], self.mode, self.rpw)

    def assert_out(self, d, ref):
        got = _h(d["out"]).reshape(self.nv, self.nout)
        if np.array_equal(got, ref):
            return
        own = self.owner()
        bad = np.nonzero(got != ref)
        shapes = sorted({own.get(int(p), "unowned position") for p in bad[1]}, key=str)
        raise AssertionError("%d wrong outputs (options %s), from matrices (np, n) = %s" % (
            bad[0].size, sorted(self.opts), shapes[:12]))


BATCHED_OPTS = [(), ("gather", "scatter"), ("xsub",), ("mode1",), ("outoff",), ("nrows",), ("ncols",), ("rpw1",),
                ("gather", "scatter", "xsub", "mode1", "outoff", "nrows", "ncols", "rpw1")]


@pytest.mark.gpu
@pytest.mark.parametrize("opts", BATCHED_OPTS, ids=lambda o: "+".join(o) or "plain")
def test_batched_gemv_exact(kh, opts):
    """k_batched_gemv over all GEMV_SHAPES; with nrows, the lead items (rows < nrows) first, then the trail items
    from nrows on without it, as ApplyInverse splits its first solve.  Reference: exact."""
    c = GemvCase(opts, seed=len(opts) * 100 + sum(map(len, opts)))
    d = c.device()
    npmax = int(c.np_.max())
    if c.nrows_lead is not None:
        lead = c.nrows_lead
        im, ir = c.items(last=lambda m: int(lead[m]))
        assert kh("kh_batched_gemv", *c.gemv_args(d, _d(im), _d(ir), d["nrows"]), len(im), npmax) == 1
        c.assert_out(d, c.expected(rows=lambda m: (0, int(lead[m]))))
        im, ir = c.items(first=lambda m: int(lead[m]))
        assert kh("kh_batched_gemv", *c.gemv_args(d, _d(im), _d(ir)), len(im), npmax) == 1
    else:
        im, ir = c.items()
        assert kh("kh_batched_gemv", *c.gemv_args(d, _d(im), _d(ir), d["nrows"]), len(im), npmax) == 1
    c.assert_out(d, c.expected())


MULTI_OPTS = [(), ("gather", "scatter"), ("xsub",), ("outoff",), ("nrows",),
              ("gather", "scatter", "xsub", "outoff", "nrows")]


@pytest.mark.gpu
@pytest.mark.parametrize("nv", [2, 3, 4])
@pytest.mark.parametrize("opts", MULTI_OPTS, ids=lambda o: "+".join(o) or "plain")
def test_batched_gemv_multi_exact(kh, nv, opts):
    """k_batched_gemv_multi (mode 0): nv vectors at leading dimensions larger than their length.
    Reference: exact."""
    c = GemvCase(opts, seed=1000 + 10 * nv + len(opts), nv=nv)
    d = c.device()
    npmax = int(c.np_.max())
    ld_in, ld_sub, ld_out = c.nin, int(c.vecOff[-1]), c.nout
    # re-lay the vectors at padded leading dimensions
    pad_in, pad_sub, pad_out = 5, 3, 9
    xin = np.full((nv, ld_in + pad_in), 7.0)
    xin[:, :ld_in] = c.xin
    d["xin"] = _d(xin.ravel())
    if c.xsub is not None:
        xs = np.full((nv, ld_sub + pad_sub), -3.0)
        xs[:, :ld_sub] = c.xsub
        d["xsub"] = _d(xs.ravel())
    d["out"] = _d(np.full((nv, ld_out + pad_out), SENTINEL).ravel())
    accepted = C.c_int(0)
    if c.nrows_lead is not None:
        im, ir = c.items(last=lambda m: int(c.nrows_lead[m]))
        rows = (lambda m: (0, int(c.nrows_lead[m])))
    else:
        im, ir = c.items()
        rows = None
    assert kh("kh_batched_gemv_multi", *c.gemv_args(d, _d(im), _d(ir), d["nrows"]), len(im), npmax, nv,
              ld_in + pad_in, ld_sub + pad_sub, ld_out + pad_out, C.byref(accepted)) == 1
    assert accepted.value == 1
    got = _h(d["out"]).reshape(nv, ld_out + pad_out)
    assert np.all(got[:, ld_out:] == SENTINEL), "written beyond the leading dimension's vector length"
    d["out"] = _d(np.ascontiguousarray(got[:, :ld_out]).ravel())
    c.assert_out(d, c.expected(rows=rows))


WARP_CTA_OPTS = [(), ("gather", "scatter"), ("outoff",), ("gather", "scatter", "outoff")]


@pytest.mark.gpu
@pytest.mark.parametrize("subset", ["all", "null", "odd"])
@pytest.mark.parametrize("opts", WARP_CTA_OPTS, ids=lambda o: "+".join(o) or "plain")
def test_small_gemv_exact(kh, opts, subset):
    """k_small_gemv (mode 0) on every shape up to np = 520 in one launch (npMax 520), for a null matList (all
    matrices), the full list and every other matrix.  Reference: exact."""
    c = GemvCase(opts, seed=2000 + len(opts) + len(subset))
    d = c.device()
    mats = list(range(c.count)) if subset != "odd" else list(range(1, c.count, 2))
    ml = None if subset == "null" else _d(np.asarray(mats, dtype=np.int32))
    accepted = C.c_int(0)
    assert kh("kh_small_gemv", *c.gemv_args(d), ml, len(mats), int(c.np_.max()), C.byref(accepted)) == 1
    assert accepted.value == 1
    chosen = set(mats)
    c.assert_out(d, c.expected(rows=lambda m: (0, int(c.n[m]) if m in chosen else 0)))


@pytest.mark.gpu
@pytest.mark.parametrize("subset", ["all", "odd"])
@pytest.mark.parametrize("opts", WARP_CTA_OPTS, ids=lambda o: "+".join(o) or "plain")
def test_cta_gemv_exact(kh, opts, subset):
    """k_cta_gemv (mode 0, one CTA per listed matrix) on every shape.  Reference: exact."""
    c = GemvCase(opts, seed=3000 + len(opts) + len(subset))
    d = c.device()
    mats = list(range(c.count)) if subset == "all" else list(range(1, c.count, 2))
    assert kh("kh_cta_gemv", *c.gemv_args(d), np.asarray(mats, dtype=np.int32), len(mats),
              int(c.np_.max())) == 1
    chosen = set(mats)
    c.assert_out(d, c.expected(rows=lambda m: (0, int(c.n[m]) if m in chosen else 0)))


@pytest.mark.gpu
def test_gemv_split_lists_like_the_separator_blocks(kh):
    """ApplyBlockDiagonal's split: np <= 64 through k_small_gemv (npMax 64), 64 < np <= 512 through k_cta_gemv,
    the rest through the slab kernel, with one index array for gather and scatter.  Reference: exact."""
    c = GemvCase(("gather", "same_gather_scatter"), seed=4000)
    d = c.device()
    small = [m for m in range(c.count) if c.np_[m] <= 64]
    mid = [m for m in range(c.count) if 64 < c.np_[m] <= 512]
    big = [m for m in range(c.count) if c.np_[m] > 512]
    accepted = C.c_int(0)
    assert kh("kh_small_gemv", *c.gemv_args(d), np.asarray(small, dtype=np.int32), len(small), 64,
              C.byref(accepted)) == 1 and accepted.value == 1
    assert kh("kh_cta_gemv", *c.gemv_args(d), np.asarray(mid, dtype=np.int32), len(mid), 512) == 1
    im, ir = c.items()
    keep = np.isin(im, big)
    assert kh("kh_batched_gemv", *c.gemv_args(d, _d(im[keep]), _d(ir[keep])), int(keep.sum()),
              int(c.np_.max())) == 1
    c.assert_out(d, c.expected())


@pytest.mark.gpu
def test_small_gemv_refuses_blocks_above_its_limit(kh):
    c = GemvCase((), seed=5000, shapes=[(8, 8)])
    d = c.device()
    accepted = C.c_int(1)
    assert kh("kh_small_gemv", *c.gemv_args(d), None, 1, 2056, C.byref(accepted)) == 0
    assert accepted.value == 0
    assert np.all(_h(d["out"]) == SENTINEL)


# ---------------------------------------------------------------------------------------------------------------
# Krylov vector kernels
# ---------------------------------------------------------------------------------------------------------------
DOT_NS = [1, 1001, 151552, 300001]  # odd and even, below and above 592 blocks x 256 threads


def _two_prod(a, b):
    """a * b = p + e exactly, elementwise (Dekker's product with Veltkamp's split): with math.fsum over p and e
    the dot product is exact up to its one final rounding."""
    def split(x):
        c = 134217729.0 * x  # 2^27 + 1
        hi = c - (c - x)
        return hi, x - hi
    p = a * b
    a1, a2 = split(a)
    b1, b2 = split(b)
    return p, ((a1 * b1 - p) + a1 * b2 + a2 * b1) + a2 * b2


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 7, 8, 9, 17, 31])
@pytest.mark.parametrize("n", DOT_NS)
@pytest.mark.parametrize("variant", ["plain", "widx_accumulate"])
def test_multi_dot(kh, k, n, variant):
    """h[i] (+)= V_i . w (optionally w[widx[r]]).  Reference: math.fsum (exact sum, one rounding).  Bound of any
    summation order: |h^ - h| <= gamma(n + 1) (|h0| + sum |v w|) (the +1 for the accumulation).  Two runs are
    bitwise equal (the summation order is fixed)."""
    import torch
    rng = np.random.default_rng([n, k, len(variant)])
    ldv = n + 3
    V = rng.standard_normal((k, ldv))
    wlen = n + 11 if variant != "plain" else n
    w = rng.standard_normal(wlen)
    widx = rng.permutation(wlen)[:n].astype(np.int32) if variant != "plain" else None
    h0 = rng.standard_normal(k) if variant != "plain" else np.full(k, np.nan)
    acc = 1 if variant != "plain" else 0
    wg = w[widx] if widx is not None else w
    nblk = 592
    dV, dw = _d(V), _d(w)
    dwidx = None if widx is None else _d(widx)
    runs = []
    for _ in range(2):
        dh = _d(h0)
        partial = torch.full((k * nblk,), float("nan"), dtype=torch.float64, device="cuda")
        assert kh("kh_multi_dot", dV, ldv, k, dw, n, partial, dh, acc, dwidx) == 2
        runs.append(_h(dh))
    assert np.array_equal(runs[0], runs[1]), "multiDot is not reproducible"
    for i in range(k):
        p, e = _two_prod(V[i, :n], wg)
        ref = math.fsum(p.tolist() + e.tolist() + ([h0[i]] if acc else []))
        tol = gamma(n + 1) * (float(np.abs(p).sum()) + (abs(h0[i]) if acc else 0.0))
        assert abs(runs[0][i] - ref) <= tol, "vector %d of %d: %.17g vs %.17g (tol %.3e)" % (i, k, runs[0][i], ref,
                                                                                            tol)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 7, 8, 9, 17])
@pytest.mark.parametrize("n", [1, 2, 1001, 200001])
@pytest.mark.parametrize("layout", ["paired", "odd_ldv", "basis_offset", "w_offset"])
@pytest.mark.parametrize("sign", [1.0, -1.0])
def test_multi_axpy_exact(kh, k, n, layout, sign):
    """w += sign sum_i h[i] V_i on the 16-byte paired path (odd n: its tail row) and on the one-row path (odd ldv,
    a basis or w one double off 16-byte alignment).  Integers: exact; entries of w beyond n stay untouched."""
    import torch
    rng = np.random.default_rng([n, k, len(layout)])
    ldv = n + 1 + n % 2 if layout == "odd_ldv" else n + 2 - n % 2  # odd / even, larger than n
    V = _ints(rng, (k, ldv))
    h = _ints(rng, k)
    w = _ints(rng, n + 3)
    vshift = 1 if layout == "basis_offset" else 0
    wshift = 1 if layout == "w_offset" else 0
    dVbuf = torch.zeros(k * ldv + 2, dtype=torch.float64, device="cuda")
    dVbuf[vshift:vshift + k * ldv] = _d(V.ravel())
    dwbuf = torch.zeros(n + 3 + 2, dtype=torch.float64, device="cuda")
    dwbuf[wshift:wshift + n + 3] = _d(w)
    ref = w.copy()
    ref[:n] += sign * (h @ V[:, :n])
    launches = kh("kh_multi_axpy", dVbuf.data_ptr() + 8 * vshift, ldv, k, h, dwbuf.data_ptr() + 8 * wshift, n,
                  sign)
    assert launches == 1
    assert np.array_equal(_h(dwbuf)[wshift:wshift + n + 3], ref)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 255, 256, 10007])
@pytest.mark.parametrize("variant", ["no_b", "b", "b_bidx"])
def test_spmv_exact(kh, n, variant):
    """y[r] = alpha b[bidx[r]] + beta sum_e val[e] x[col[e]], with empty rows.  Integers: exact."""
    rng = np.random.default_rng([n, len(variant)])
    ncol = n + 13
    counts = rng.integers(0, 7, n)
    counts[::5] = 0
    ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    val, col = _ints(rng, int(ptr[-1])), rng.integers(0, ncol, int(ptr[-1])).astype(np.int32)
    S = sp.csr_matrix((val, col, ptr), shape=(n, ncol))  # repeated columns are summed, by scipy and by the kernel
    x = _ints(rng, ncol)
    b = _ints(rng, n + 20) if variant != "no_b" else None
    bidx = rng.permutation(n + 20)[:n].astype(np.int32) if variant == "b_bidx" else None
    alpha, beta = (2.0, -1.0) if variant != "no_b" else (5.0, 3.0)
    ref = beta * (S @ x)
    if b is not None:
        ref = alpha * (b[bidx] if bidx is not None else b[:n]) + ref
    y = _d(np.full(n + 4, SENTINEL))
    launches = kh("kh_spmv", ptr, col, val,
                  x, y, n, alpha, b, bidx,
                  beta)
    assert launches == 1
    assert np.array_equal(_h(y), np.concatenate([ref, np.full(4, SENTINEL)]))


# ---------------------------------------------------------------------------------------------------------------
# Householder transforms of the separator groups (apply.cu k_householder)
# ---------------------------------------------------------------------------------------------------------------
HH_LENGTHS = [1, 2, 31, 32, 33, 64, 65, 100, 257, 5]


@pytest.mark.gpu
@pytest.mark.parametrize("vsum_in", [False, True])
@pytest.mark.parametrize("vsum_out", [False, True])
@pytest.mark.parametrize("export", [False, True])
@pytest.mark.parametrize("in_place", [False, True])
def test_householder(kh, vsum_in, vsum_out, export, in_place):
    """out = 2 w (w^T v) - v per group (v with its first entry replaced by vsumIn[u] when given), groups longer
    than a warp, one group with w = 0 (H = -I).  Reference: longdouble.  Per entry p of a group of m entries,
    with S = sum |w v| and t = w^T v:  |out^ - out| <= 2 |w_p| gamma(m) S + gamma(2) (2 |w_p| (|t| + gamma(m) S)
    + |v_p|) (the sum t, then one multiply and one subtract)."""
    import torch
    rng = np.random.default_rng([int(vsum_in), int(vsum_out), int(export), int(in_place)])
    starts = np.concatenate([[0], np.cumsum(HH_LENGTHS)]).astype(np.int32)
    P, nuniq = int(starts[-1]), len(HH_LENGTHS)
    w = rng.standard_normal(P)
    for u in range(nuniq):
        seg = slice(starts[u], starts[u + 1])
        w[seg] /= np.linalg.norm(w[seg])
    w[starts[3]:starts[4]] = 0.0
    v_in = rng.standard_normal(P)
    vsin = rng.standard_normal(nuniq) if vsum_in else None
    Xlen = P + 17
    sepRow = rng.permutation(Xlen)[:P].astype(np.int32) if export else None
    # reference
    v = v_in.copy()
    if vsum_in:
        v[starts[:-1]] = vsin
    ref = np.empty(P, dtype=LD)
    tol = np.empty(P)
    for u in range(nuniq):
        seg = slice(starts[u], starts[u + 1])
        m = HH_LENGTHS[u]
        t = np.sum(w[seg].astype(LD) * v[seg].astype(LD))
        S = float(np.abs(w[seg] * v[seg]).sum())
        ref[seg] = 2 * w[seg].astype(LD) * t - v[seg].astype(LD)
        tol[seg] = 2 * np.abs(w[seg]) * gamma(m) * S + gamma(2) * (2 * np.abs(w[seg]) * (abs(float(t)) + gamma(m) * S)
                                                                   + np.abs(v[seg]))
    din = _d(v_in)
    dout = din if in_place else torch.full_like(din, float("nan"))
    dvso = _d(np.full(nuniq, SENTINEL)) if vsum_out else None
    dX = _d(np.full(Xlen, SENTINEL)) if export else None
    launches = kh("kh_householder", starts, nuniq, w, din, dout, dvso,
                  vsin, dX, sepRow)
    assert launches == 1
    out = _h(dout)
    err = np.abs((out.astype(LD) - ref).astype(np.float64))
    assert np.all(err <= tol), "entries %s off by %s (tol %s)" % (np.nonzero(err > tol)[0][:5], err[err > tol][:5],
                                                                  tol[err > tol][:5])
    if vsum_out:
        assert np.array_equal(_h(dvso), out[starts[:-1]])
    if export:
        X = _h(dX)
        assert np.array_equal(X[sepRow], out)
        untouched = np.ones(Xlen, dtype=bool)
        untouched[sepRow] = False
        assert np.all(X[untouched] == SENTINEL)
