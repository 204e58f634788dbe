"""The "Krylov Basis Precision" parameter of the "Solver" sublist ("Double", the default, or "Single": FP32 storage of
the GMRES basis vectors after the first of each cycle, FP64 arithmetic).  Its rules are host work, checked here without
a GPU: the accepted values, the rejection of any other value and of Single with CG at create and at SetParameters
(which keeps the old list), and the final list of a run that does not name it."""
import pytest

import hymls_b200 as hb

ERR_ARG = -1
NAME = "Krylov Basis Precision"


def _params(precision=None, method=None, solver=True):
    p = {"Problem": {"Equations": "Stokes-C", "Dimension": 3, "nx": 16, "ny": 16, "nz": 16},
         "Preconditioner": {"Partitioner": "Skew Cartesian", "Separator Length": 4, "Number of Levels": 2,
                            "Coarsening Factor": 2}}
    if solver:
        p["Solver"] = {"Iterative Solver": {"Num Blocks": 20}}
        if precision is not None:
            p["Solver"][NAME] = precision
        if method is not None:
            p["Solver"]["Krylov Method"] = method
    return p


def _final(P):
    from hymls_b200 import driver
    return driver.parse_parameter_list(P.GetParametersXml())


@pytest.mark.parametrize("value", ["Single", "Double"])
def test_single_and_double_are_accepted(value):
    P = hb.Preconditioner(None, _params(value))
    assert _final(P)["Solver"][NAME] == value
    P.SetParameters(_params(value, method="GMRES"))
    assert _final(P)["Solver"][NAME] == value


def test_double_is_accepted_with_cg():
    P = hb.Preconditioner(None, _params("Double", method="CG"))
    assert _final(P)["Solver"][NAME] == "Double"


@pytest.mark.parametrize("value", ["Half", "single", 1, True])
def test_other_values_are_rejected_at_create(value):
    with pytest.raises(hb.HymlsError) as e:
        hb.Preconditioner(None, _params(value))
    assert e.value.code == ERR_ARG


def test_single_with_cg_is_rejected():
    with pytest.raises(hb.HymlsError) as e:
        hb.Preconditioner(None, _params("Single", method="CG"))
    assert e.value.code == ERR_ARG
    P = hb.Preconditioner(None, _params("Double", method="CG"))
    before = P.GetParametersXml()
    with pytest.raises(hb.HymlsError) as e:
        P.SetParameters(_params("Single", method="CG"))
    assert e.value.code == ERR_ARG and P.GetParametersXml() == before


@pytest.mark.parametrize("value", ["Half", 1])
def test_set_parameters_rejects_and_keeps_the_old_list(value):
    P = hb.Preconditioner(None, _params("Single"))
    before = P.GetParametersXml()
    with pytest.raises(hb.HymlsError) as e:
        P.SetParameters(_params(value))
    assert e.value.code == ERR_ARG
    assert P.GetParametersXml() == before and _final(P)["Solver"][NAME] == "Single"


def test_the_default_is_not_written_back():
    A = -hb.galeri.create_matrix("Stokes-C", 3, 16)
    P = hb.Preconditioner(A, _params(), pattern_only=True)
    P.Initialize()
    assert NAME not in P.GetParametersXml()
    assert "Num Blocks" in P.GetParametersXml()


def test_no_solver_sublist_is_added():
    A = -hb.galeri.create_matrix("Stokes-C", 3, 16)
    P = hb.Preconditioner(A, _params(solver=False), pattern_only=True)
    P.Initialize()
    P.SetParameters(_params(solver=False))
    assert "Solver" not in _final(P) and NAME not in P.GetParametersXml()


def test_basis_bytes_are_zero_before_a_solve():
    A = -hb.galeri.create_matrix("Stokes-C", 3, 16)
    for value in (None, "Single"):
        P = hb.Preconditioner(A, _params(value), pattern_only=True)
        P.Initialize()
        assert P.Stats()["krylov_basis_bytes"] == 0
