"""The host dense eigensolver of the GCRO-DR restart (hymls_b200/csrc/dense_eig.cpp), compiled alone with g++ and called
through ctypes: eigenvalues and eigenvectors against numpy / scipy, the harmonic Ritz selection (complex pairs kept
whole) against the generalized eigenproblem solved by QZ, the Householder QR, and the rank-deficient fallback."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import scipy.linalg as sl

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_dp = np.ctypeslib.ndpointer(dtype=np.float64, flags="F_CONTIGUOUS")
_ip = C.POINTER(C.c_int)


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("dense_eig") / "dense_eig.so")
    src = os.path.join(ROOT, "hymls_b200", "csrc", "dense_eig.cpp")
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-Werror", "-fPIC", "-shared", src, "-o", so],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    L = C.CDLL(so)
    L.hy_eig.argtypes = [C.c_int, _dp, _dp, _dp, _dp]
    L.hy_qr.argtypes = [C.c_int, C.c_int, _dp, _dp, _dp, C.c_double]
    L.hy_harmonic_ritz.argtypes = [C.c_int, _dp, _dp, C.c_int, C.c_int, _dp, _ip]
    for f in (L.hy_eig, L.hy_qr, L.hy_harmonic_ritz):
        f.restype = C.c_int
    return L


def _f(a):
    return np.asfortranarray(a, dtype=np.float64)


def _eig(lib, A):
    n = A.shape[0]
    wr, wi, V = _f(np.zeros((n, 1))), _f(np.zeros((n, 1))), _f(np.zeros((n, n)))
    assert lib.hy_eig(n, _f(A), wr, wi, V) == 0
    lam = wr[:, 0] + 1j * wi[:, 0]
    X = V.astype(complex)
    j = 0
    while j < n:   # pair: columns j, j+1 = real and imaginary part of the vector of lam[j] (wi > 0)
        if wi[j, 0] != 0:
            assert wi[j, 0] > 0 and lam[j + 1] == np.conj(lam[j])
            X[:, j] = V[:, j] + 1j * V[:, j + 1]
            X[:, j + 1] = V[:, j] - 1j * V[:, j + 1]
            j += 2
        else:
            j += 1
    return lam, X


def _matrices():
    rng = np.random.default_rng(3)
    out = {}
    for n in (1, 2, 3, 64, 600):
        out["random%d" % n] = rng.standard_normal((n, n))
    out["hessenberg64"] = np.triu(rng.standard_normal((64, 64)), -1)
    R = np.array([[0.0, 2.0], [-2.0, 0.0]])   # rotation blocks: eigenvalues +-2i, and more pairs
    Q, _ = np.linalg.qr(rng.standard_normal((6, 6)))
    out["pairs6"] = Q @ sl.block_diag(R, [[1.0, 5.0], [-0.2, 1.0]], [[3.0]], [[-1.0]]) @ Q.T
    out["repeated8"] = Q @ np.diag([2.0, 2.0, 2.0, -1.0, -1.0, 0.5]) @ Q.T
    J = np.diag(np.full(5, 1.5)) + np.diag(np.ones(4), 1)   # one Jordan block: defective
    out["jordan5"] = J
    out["zero4"] = np.zeros((4, 4))
    out["triangular5"] = np.triu(rng.standard_normal((5, 5)))
    return out


MATS = _matrices()
DEFECTIVE = {"jordan5": 5}


@pytest.mark.parametrize("name", sorted(MATS))
def test_eigenpairs_against_numpy(lib, name):
    A = MATS[name]
    n = A.shape[0]
    lam, X = _eig(lib, A)
    nrmA = max(np.linalg.norm(A, 2), 1e-300)
    # residuals of the eigenpairs
    for j in range(n):
        v = X[:, j]
        if name in DEFECTIVE:
            continue
        assert np.linalg.norm(A @ v - lam[j] * v) <= 1e-12 * nrmA * np.linalg.norm(v) + 1e-300
    # eigenvalues: every numpy eigenvalue has one of ours within 1e-12 ||A|| times its condition number
    ref, VL, VR = sl.eig(A, left=True, right=True)
    used = np.zeros(n, bool)
    for i in np.argsort(-np.abs(ref)):
        if name in DEFECTIVE:
            tol = 4 * (np.finfo(float).eps * nrmA) ** (1.0 / DEFECTIVE[name]) * max(nrmA, 1.0)
        else:
            y, x = VL[:, i], VR[:, i]
            cond = np.linalg.norm(y) * np.linalg.norm(x) / max(abs(np.vdot(y, x)), 1e-300)
            tol = 1e-12 * nrmA * max(cond, 1.0) + 1e-300
        d = np.where(used, np.inf, np.abs(lam - ref[i]))
        j = int(np.argmin(d))
        assert d[j] <= tol, (name, ref[i], lam[j], tol)
        used[j] = True


def test_eig_is_deterministic(lib):
    A = MATS["random64"]
    a, b = _eig(lib, A), _eig(lib, A)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@pytest.mark.parametrize("m,n", [(1, 1), (5, 3), (31, 30), (601, 40)])
def test_qr(lib, m, n):
    A = np.random.default_rng(m + n).standard_normal((m, n))
    Q, R = _f(np.zeros((m, n))), _f(np.zeros((n, n)))
    assert lib.hy_qr(m, n, _f(A), Q, R, 1e-14) == 0
    assert np.allclose(Q @ R, A, rtol=0, atol=1e-13 * np.linalg.norm(A))
    assert np.allclose(Q.T @ Q, np.eye(n), rtol=0, atol=1e-13)
    assert np.all(np.diag(R) > 0) and np.array_equal(R, np.triu(R))


def test_qr_reports_rank_deficiency(lib):
    A = np.random.default_rng(1).standard_normal((20, 4))
    A[:, 3] = A[:, 0] - 2 * A[:, 1]
    Q, R = _f(np.zeros((20, 4))), _f(np.zeros((4, 4)))
    assert lib.hy_qr(20, 4, _f(A), Q, R, 1e-12) == 1


def _ritz(lib, A, B, k, kmax):
    n = A.shape[0]
    P = _f(np.zeros((n, kmax)))
    kout = C.c_int(-1)
    rc = lib.hy_harmonic_ritz(n, _f(A), _f(B), k, kmax, P, C.byref(kout))
    return rc, P[:, :kout.value]


def _oracle_selection(A, B, k):
    """QZ on (A, B): the k smallest |theta| (pairs whole) and the span of their vectors"""
    th, Z = sl.eig(A, B)
    mod = np.where(np.isfinite(th), np.abs(th), np.inf)
    order = np.argsort(mod, kind="stable")
    sel = list(order[:k])
    for i in list(sel):
        if abs(th[i].imag) > 0:
            j = int(np.argmin(np.where(np.arange(len(th)) == i, np.inf, np.abs(th - np.conj(th[i])))))
            if j not in sel:
                sel.append(j)
    Zs = Z[:, sel]
    return th[sel], np.hstack([Zs.real, Zs.imag])


def _gen_problem(seed, mt):
    """A = G'G, B = G'[I; 0] (the first-cycle harmonic problem of a Hessenberg G)"""
    rng = np.random.default_rng(seed)
    G = np.triu(rng.standard_normal((mt + 1, mt)), -1) + 3 * np.eye(mt + 1, mt)
    return G.T @ G, G.T @ np.eye(mt + 1, mt)


@pytest.mark.parametrize("seed,mt,k", [(0, 10, 3), (1, 30, 5), (2, 60, 20), (3, 8, 1)])
def test_harmonic_ritz_against_qz(lib, seed, mt, k):
    A, B = _gen_problem(seed, mt)
    rc, P = _ritz(lib, A, B, k, k + 1)
    assert rc == 0 and P.shape[1] in (k, k + 1)
    th, Zs = _oracle_selection(A, B, k)
    assert P.shape[1] == len(th)
    # the same space: the columns of P satisfy A P = B P Theta within the selected subspace of the oracle
    Qo = sl.orth(Zs)
    assert Qo.shape[1] == P.shape[1]
    Qp, _ = np.linalg.qr(P)
    s = np.linalg.svd(Qo.T @ Qp, compute_uv=False)
    assert s.min() > 1 - 1e-8, s


def test_conjugate_pair_straddling_k(lib):
    # theta = 1/mu; S = diag(4, rot(3, 1)=3+-i, 0.5): |mu| order 4, |3+-i|, ... -> k = 2 straddles the pair
    rot = np.array([[3.0, 1.0], [-1.0, 3.0]])
    S = sl.block_diag([[4.0]], rot, [[0.5]], [[0.25]])
    A = np.eye(5)
    B = S                      # L = I: S = B, mu = eig(S)
    rc, P = _ritz(lib, A, B, 2, 3)
    assert rc == 0 and P.shape[1] == 3
    th, Zs = _oracle_selection(A, B, 2)   # theta = 1/mu: smallest |theta| = largest |mu|
    assert len(th) == 3
    span = sl.orth(Zs)
    assert np.linalg.norm(P - span @ (span.T @ P)) <= 1e-12 * np.linalg.norm(P)
    # no room for k + 1: the pair is left out
    rc, P = _ritz(lib, A, B, 2, 2)
    assert rc == 0 and P.shape[1] == 1
    assert abs(abs(P[0, 0]) - np.linalg.norm(P)) < 1e-14 * np.linalg.norm(P)


def test_rank_deficient_problem_is_refused(lib):
    rng = np.random.default_rng(4)
    G = rng.standard_normal((9, 8))
    G[:, 5] = G[:, 2]          # rank-deficient G: G'G is singular, its Cholesky factorisation fails
    rc, P = _ritz(lib, G.T @ G, G.T @ np.eye(9, 8), 3, 4)
    assert rc == 1 and P.shape[1] == 0
