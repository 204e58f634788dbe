"""The driver flow of `hymls_main <params.xml>` (src/main.cpp:48-535) on the shipped configurations:
configs/*.xml are BASELINE.json's five configurations with the reference's parameter names."""
import glob
import os

import numpy as np
import pytest
import scipy.sparse as sp

import hymls_b200 as hb
from hymls_b200 import driver
from tests.conftest import ROOT

CONFIGS = sorted(glob.glob(os.path.join(ROOT, "configs", "*.xml")))


def test_configs_parse_and_validate_on_cpu():
    assert len(CONFIGS) == 5
    for f in CONFIGS:
        xml = open(f).read()
        p = driver.parse_parameter_list(xml)
        assert {"Problem", "Solver", "Preconditioner"} <= set(p)
        hb.Preconditioner(None, xml)          # C-side XML parser + parameter validation (no device needed)


def test_stale_reference_parameter_is_rejected_like_validate_parameters():
    xml = open(os.path.join(ROOT, "configs", "cavity.xml")).read().replace(
        '<Parameter name="Partitioner"', '<Parameter name="Classifier" type="string" value="Stokes"/>\n'
        '<Parameter name="Partitioner"')
    with pytest.raises(hb.HymlsError) as e:   # src/HYMLS_Preconditioner.cpp:126-130
        hb.Preconditioner(None, xml)
    assert "Classifier" in str(e.value)


def test_nullspace_generators():
    prob = {"Equations": "Stokes-C", "Dimension": 2, "nx": 4, "ny": 4}
    V = driver.create_nullspace(48, "Constant P", prob)
    assert V.shape == (48, 1) and np.allclose(np.linalg.norm(V, axis=0), 1)
    assert np.all(V[2::3, 0] > 0) and np.all(V[0::3, 0] == 0) and np.all(V[1::3, 0] == 0)
    C = driver.create_nullspace(48, "Checkerboard", prob)
    assert C.shape == (48, 2) and abs(C[:, 0] @ C[:, 1]) < 1e-15
    assert np.allclose(C[2::3].sum(axis=1), C[2, :].sum())
    K = driver.create_nullspace(48, "Constant", prob)
    assert K.shape == (48, 3) and np.allclose(K.T @ K, np.eye(3))


GPU_RUNS = [
    ("laplace.xml", {"Problem/nx": 64, "Problem/ny": 64}, 35, 1e-9),
    ("stokes2D.xml", {"Problem/nx": 64, "Problem/ny": 64}, 200, 1e-9),
    ("cavity.xml", {}, 250, 1e-10),
    ("cavity3D.xml", {"Problem/nx": 16, "Problem/ny": 16, "Problem/nz": 16, "Preconditioner/Separator Length": 4,
                      "Preconditioner/Coarsening Factor": 2}, 200, 1e-7),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,over,max_its,tol", GPU_RUNS, ids=[r[0] for r in GPU_RUNS])
def test_configs_run_on_gpu(name, over, max_its, tol):
    out = driver.run(open(os.path.join(ROOT, "configs", name)).read(), over, verbose=False)
    assert out["converged"] and out["iterations"] <= max_its
    assert out["residual"] <= tol
    if name == "cavity.xml":   # fixture solution available: error with the constant pressure projected out
        assert out["border"] == 1 and out["levels"] == 3
        assert out["error"] <= 1e-8


def test_final_parameter_list_round_trip():
    """'Store Final Parameter List' (src/main.cpp:492-509): the list with the defaults the partitioner wrote
    back (SetParameters, src/HYMLS_BasePartitioner.cpp:31-319) comes out as Teuchos XML and reproduces the run."""
    import scipy.sparse as sp
    from tests.conftest import load_fixture
    A, _, _ = load_fixture("cavity2d_32_Re1000")
    xml = open(os.path.join(ROOT, "configs", "cavity.xml")).read()
    P = hb.Preconditioner(sp.csr_matrix(A), xml, pattern_only=True)
    P.Initialize()
    final = driver.parse_parameter_list(P.GetParametersXml())
    assert final["Problem"]["Degrees of Freedom"] == 3 and final["Problem"]["Pressure Variable"] == 2
    assert final["Problem"]["Variable 2"]["Variable Type"] == "Pressure"
    assert final["Preconditioner"]["Eliminate Velocities Together"] is True
    assert final["Preconditioner"]["Number of Levels"] == 3 and final["Driver"]["Null Space Type"] == "Constant P"
    hb.Solver(P).SetTolerance(1e-6)               # BaseSolver::SetTolerance, what NOX calls before every solve
    assert driver.parse_parameter_list(P.GetParametersXml())["Solver"]["Iterative Solver"][
        "Convergence Tolerance"] == 1e-6
    with pytest.raises(hb.HymlsError):
        hb.Solver(P).SetTolerance(-1.0)
    Q = hb.Preconditioner(sp.csr_matrix(A), P.GetParametersXml(), pattern_only=True)
    Q.Initialize()
    assert Q.NumLevels() == P.NumLevels()
    for lev in range(P.NumLevels()):
        assert np.array_equal(P.GetMap(hb.api.MAP_SEPARATOR, lev), Q.GetMap(hb.api.MAP_SEPARATOR, lev))


def test_parameter_list_xml_details():
    xml = """<!-- leading comment -->
    <ParameterList name="HYMLS"><!--{-->
      <ParameterList name="Problem">
        <Parameter value="8" name="nx" type="int"/>   <!-- attribute order is free -->
        <Parameter name="Equations" type="string" value="Laplace"/>
        <Parameter name="Dimension" type="int" value="2"/>
      </ParameterList>
      <ParameterList name="Preconditioner">
        <Parameter name="Separator Length" type="int" value="4"/>
        <Parameter name="Fix Pressure Level" type="bool" value="0"/>
        <Parameter name="Apply Dropping" type="bool" value="true"/>
        <ParameterList name="Coarse Solver">
          <Parameter name="amesos: solver type" type="string" value="Amesos_Klu &amp; friends"/>
        </ParameterList>
      </ParameterList>
    </ParameterList>"""
    P = hb.Preconditioner(None, xml)
    out = driver.parse_parameter_list(P.GetParametersXml())
    assert out["Problem"]["nx"] == 8 and out["Preconditioner"]["Fix Pressure Level"] is False
    assert out["Preconditioner"]["Coarse Solver"]["amesos: solver type"] == "Amesos_Klu & friends"
    with pytest.raises(hb.HymlsError):
        hb.Preconditioner(None, "<ParameterList name='x'><Parameter name='a' type='int' value='1'/>")  # not closed


class _OraclePrec:
    """Stand-in for hymls_b200.Preconditioner backed by the numpy ORACLE: lets the hymls_main flow of
    hymls_b200/driver.py (factorization / solve loops, diagonal perturbation) run on a machine without a GPU.
    Test infrastructure only."""
    log = []

    def __init__(self, K, params, tv):
        from oracle import hymls as oh
        from oracle.params import ParameterList

        def to_pl(d):
            pl = ParameterList()
            for k, v in d.items():
                pl[k] = to_pl(v) if isinstance(v, dict) else v
            return pl
        self._mk = lambda K_: oh.Preconditioner(K_, to_pl(params), tv)
        self.K = K
        self.O = self._mk(K)
        _OraclePrec.log.append("create")

    def Initialize(self):
        self.O.initialize()
        _OraclePrec.log.append("Initialize")

    def SetMatrix(self, K):
        assert np.array_equal(K.indptr, self.K.indptr) and np.array_equal(K.indices, self.K.indices)  # same pattern
        self.K = K
        self.O = self._mk(K)
        self.O.initialize()
        _OraclePrec.log.append("SetMatrix")

    def Compute(self):
        self.O.compute()
        _OraclePrec.log.append("Compute")

    def NumLevels(self):
        return 1

    def NumMySubdomains(self, level):
        return len(self.O.hid.interior)


class _OracleSolver:
    def __init__(self, P):
        self.P = P

    def ApplyInverse(self, b, seed=0):
        from oracle import krylov as ok
        K, O = self.P.K, self.P.O
        x, its, conv, h = ok.cg(lambda v: K @ v, b, np.zeros(len(b)), O.apply_inverse, tol=1e-10, max_iters=200)
        self.num_iter, self.history = its, h
        self.info = {"converged": conv, "solve_seconds": 0.0}
        _OraclePrec.log.append("Solve")
        return x


def test_driver_factorization_and_solve_loops(monkeypatch):
    """hymls_main's "Number of factorizations" x "Number of solves" loops with a "Diagonal Perturbation"
    (src/main.cpp:341-470): Initialize once, then per factorization SetMatrix (same pattern) + Compute and the
    solves, each with a fresh right-hand side."""
    from hymls_b200 import driver
    monkeypatch.setattr(driver, "Preconditioner", _OraclePrec)
    monkeypatch.setattr(driver, "Solver", _OracleSolver)
    _OraclePrec.log = []
    xml = open(os.path.join(ROOT, "configs", "laplace.xml")).read()
    over = {"Problem/nx": 16, "Problem/ny": 16, "Preconditioner/Number of Levels": 1,
            "Driver/Number of factorizations": 2, "Driver/Number of solves": 3, "Driver/Diagonal Perturbation": 0.05}
    out = driver.run(xml, over, verbose=False)
    assert _OraclePrec.log == ["create", "Initialize"] + (["SetMatrix", "Compute"] + ["Solve"] * 3) * 2
    assert [(r["factorization"], r["solve"]) for r in out["runs"]] == [(f, s) for f in (1, 2) for s in (1, 2, 3)]
    assert all(r["converged"] and r["residual"] < 1e-9 and r["error"] < 1e-8 for r in out["runs"])
    K = out["_objects"][0]
    K0 = hb.galeri.create_matrix("Laplace", 2, 16)
    d = K.diagonal() - K0.diagonal()
    assert 0 < np.abs(d).max() <= 0.05 and (K - K0 - sp.diags(d)).nnz == 0    # only the diagonal moved
    # defaults: one factorization, one solve, no SetMatrix -- the flow the GPU tests run
    _OraclePrec.log = []
    out1 = driver.run(xml, {"Problem/nx": 16, "Problem/ny": 16, "Preconditioner/Number of Levels": 1}, verbose=False)
    assert _OraclePrec.log == ["create", "Initialize", "Compute", "Solve"] and len(out1["runs"]) == 1
    assert out1["iterations"] == out1["runs"][0]["iterations"] and out1["residual"] < 1e-9
