"""The GCRO-DR parameters of the "Solver" sublist ("Krylov Method" = "GCRODR", "Iterative Solver" / "Num Recycled
Blocks"): the rejections at create and at SetParameters (which keeps the old list), and lists that do not select
GCRODR read back unchanged.  Host work, checked without a GPU."""
import pytest

import hymls_b200 as hb

ERR_ARG = -1
NAME = "Num Recycled Blocks"


def _params(method="GCRODR", k=None, blocks=20, precision=None):
    p = {"Problem": {"Equations": "Stokes-C", "Dimension": 3, "nx": 16, "ny": 16, "nz": 16},
         "Preconditioner": {"Partitioner": "Skew Cartesian", "Separator Length": 4, "Number of Levels": 2,
                            "Coarsening Factor": 2},
         "Solver": {"Krylov Method": method, "Iterative Solver": {}}}
    if blocks is not None:
        p["Solver"]["Iterative Solver"]["Num Blocks"] = blocks
    if k is not None:
        p["Solver"]["Iterative Solver"][NAME] = k
    if precision is not None:
        p["Solver"]["Krylov Basis Precision"] = precision
    return p


def _final(P):
    from hymls_b200 import driver
    return driver.parse_parameter_list(P.GetParametersXml())


@pytest.mark.parametrize("k", [1, 5, 19])
def test_valid_lists_are_accepted(k):
    P = hb.Preconditioner(None, _params(k=k))
    assert _final(P)["Solver"]["Iterative Solver"][NAME] == k
    P.SetParameters(_params(k=k, blocks=None))
    assert _final(P)["Solver"]["Iterative Solver"][NAME] == k


BAD = {"single_basis": dict(k=5, precision="Single"), "non_integer": dict(k=5.5), "string": dict(k="5"),
       "bool": dict(k=True), "zero": dict(k=0), "negative": dict(k=-3), "equal_to_num_blocks": dict(k=20),
       "above_num_blocks": dict(k=40)}


@pytest.mark.parametrize("case", sorted(BAD))
def test_rejected_at_create(case):
    with pytest.raises(hb.HymlsError) as e:
        hb.Preconditioner(None, _params(**BAD[case]))
    assert e.value.code == ERR_ARG


@pytest.mark.parametrize("case", sorted(BAD))
def test_rejected_at_set_parameters_keeping_the_old_list(case):
    P = hb.Preconditioner(None, _params(k=3))
    before = P.GetParametersXml()
    with pytest.raises(hb.HymlsError) as e:
        P.SetParameters(_params(**BAD[case]))
    assert e.value.code == ERR_ARG
    assert P.GetParametersXml() == before


def test_the_value_is_not_checked_for_other_methods():
    for method in ("GMRES", "CG"):
        hb.Preconditioner(None, _params(method=method, k=40))


@pytest.mark.parametrize("method", ["GMRES", "CG"])
def test_other_methods_get_no_num_recycled_blocks(method):
    A = -hb.galeri.create_matrix("Stokes-C", 3, 16)
    P = hb.Preconditioner(A, _params(method=method), pattern_only=True)
    P.Initialize()
    assert NAME not in P.GetParametersXml()
    P.SetParameters(_params(method=method))
    assert NAME not in P.GetParametersXml()


def test_gcrodr_list_without_the_value_gets_no_default_before_a_solve():
    A = -hb.galeri.create_matrix("Stokes-C", 3, 16)
    P = hb.Preconditioner(A, _params(), pattern_only=True)
    P.Initialize()
    assert NAME not in P.GetParametersXml()
    assert P.Stats()["krylov_recycle_dim"] == 0
