"""Self-tests of the GCRO-DR restatement (tests/gcrodr_reference.py) on small problems without a GPU: its first cycle
is GMRES, recycling helps later right-hand sides, and GCRODR(m, k) beats GMRES(m)."""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle.krylov import gmres
from tests.gcrodr_reference import gcrodr


def _convection_diffusion(n, c=20.0):
    """upwind convection-diffusion on the unit square, n x n interior points (nonsymmetric)"""
    h = 1.0 / (n + 1)
    L = sp.diags([-np.ones(n - 1), 2 * np.ones(n), -np.ones(n - 1)], [-1, 0, 1]) / h ** 2
    Cx = sp.diags([-np.ones(n - 1), np.ones(n)], [-1, 0]) / h
    eye = sp.eye(n)
    return (sp.kron(eye, L) + sp.kron(L, eye) + c * sp.kron(eye, Cx) + 0.5 * c * sp.kron(Cx, eye)).tocsr()


A = _convection_diffusion(30)
N = A.shape[0]


def _op(v):
    return A @ v


def _jacobi(v):
    return v / A.diagonal()


@pytest.mark.parametrize("side", ["Right", "Left", "None"])
def test_first_cycle_is_gmres(side):
    b = np.random.default_rng(1).standard_normal(N)
    M = None if side == "None" else _jacobi
    x, it, conv, h = gmres(_op, b, np.zeros(N), apply_M=M, side=side, num_blocks=400, max_restarts=0)
    xg, itg, convg, hg, U, C = gcrodr(_op, b, np.zeros(N), apply_M=M, side=side, num_blocks=400, num_recycled=5,
                                      max_restarts=0)
    assert conv and convg and it == itg
    assert np.max(np.abs(np.array(h) - np.array(hg))) <= 1e-12
    assert U.shape[1] in (5, 6) and np.allclose(C.T @ C, np.eye(C.shape[1]), atol=1e-10)


@pytest.mark.parametrize("m,k", [(20, 5), (30, 10)])
def test_recycling_helps_later_right_hand_sides(m, k):
    rng = np.random.default_rng(2)
    its = []
    U = C = None
    for _ in range(3):
        b = rng.standard_normal(N)
        x, it, conv, h, U, C = gcrodr(_op, b, np.zeros(N), num_blocks=m, num_recycled=k, max_restarts=200,
                                      U0=U, C0=C)
        assert conv and np.linalg.norm(b - A @ x) / np.linalg.norm(b) <= 1.5e-8
        its.append(it)
    assert its[1] < its[0] and its[2] < its[0], its


@pytest.mark.parametrize("m,k", [(20, 5), (30, 10)])
def test_gcrodr_needs_fewer_iterations_than_gmres(m, k):
    b = np.random.default_rng(3).standard_normal(N)
    _, it, conv, _ = gmres(_op, b, np.zeros(N), num_blocks=m, max_restarts=200)
    _, itg, convg, _, _, _ = gcrodr(_op, b, np.zeros(N), num_blocks=m, num_recycled=k, max_restarts=200)
    assert conv and convg and itg < it, (itg, it)


def test_rebuilt_space_equals_the_kept_one():
    """U0 without C0 rebuilds C = A U0 and orthonormalises it: the same solve as with the kept C"""
    rng = np.random.default_rng(4)
    _, _, _, _, U, C = gcrodr(_op, rng.standard_normal(N), np.zeros(N), num_blocks=20, num_recycled=5,
                              max_restarts=200)
    b = rng.standard_normal(N)
    a = gcrodr(_op, b, np.zeros(N), num_blocks=20, num_recycled=5, max_restarts=200, U0=U, C0=C)
    r = gcrodr(_op, b, np.zeros(N), num_blocks=20, num_recycled=5, max_restarts=200, U0=U)
    assert a[1] == r[1]
    assert np.allclose(a[3], r[3], rtol=1e-6, atol=1e-14)
