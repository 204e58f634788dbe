"""The "Subdomain Inverse Precision" parameter of the "Preconditioner" sublist ("Double", the default, or "Single":
FP32 storage of the subdomain inverses A11^-1, FP64 arithmetic).  Its rules are host work, checked here without a GPU:
the accepted values, the rejection of any other value at create and at SetParameters (which keeps the old list), the
final list of a run that does not name it, and the A11 byte counts of the statistics after a pattern-only Initialize."""
import numpy as np
import pytest

import hymls_b200 as hb

ERR_ARG = -1
NAME = "Subdomain Inverse Precision"


def _params(precision=None):
    prec = {"Partitioner": "Skew Cartesian", "Separator Length": 4, "Number of Levels": 2, "Coarsening Factor": 2}
    if precision is not None:
        prec[NAME] = precision
    return {"Problem": {"Equations": "Stokes-C", "Dimension": 3, "nx": 16, "ny": 16, "nz": 16}, "Preconditioner": prec}


def _value(P):
    from hymls_b200 import driver
    return driver.parse_parameter_list(P.GetParametersXml())["Preconditioner"].get(NAME)


@pytest.mark.parametrize("value", ["Single", "Double"])
def test_single_and_double_are_accepted(value):
    P = hb.Preconditioner(None, _params(value))
    assert _value(P) == value
    P.SetParameters(_params(value))
    assert _value(P) == value


@pytest.mark.parametrize("value", ["Half", "single", 1, 4.0, True])
def test_other_values_are_rejected_at_create(value):
    with pytest.raises(hb.HymlsError) as e:
        hb.Preconditioner(None, _params(value))
    assert e.value.code == ERR_ARG


@pytest.mark.parametrize("value", ["Half", 1])
def test_set_parameters_rejects_and_keeps_the_old_list(value):
    P = hb.Preconditioner(None, _params("Single"))
    before = P.GetParametersXml()
    with pytest.raises(hb.HymlsError) as e:
        P.SetParameters(_params(value))
    assert e.value.code == ERR_ARG
    assert P.GetParametersXml() == before and _value(P) == "Single"


def test_the_default_is_not_written_back():
    A = -hb.galeri.create_matrix("Stokes-C", 3, 16)
    P = hb.Preconditioner(A, _params(), pattern_only=True)
    P.Initialize()
    xml = P.GetParametersXml()
    assert NAME not in xml
    assert "Separator Length" in xml           # (the other defaults are written back as before)


def test_single_counts_four_bytes_per_a11_entry():
    A = -hb.galeri.create_matrix("Stokes-C", 3, 16)
    st = {}
    for value in (None, "Double", "Single"):
        P = hb.Preconditioner(A, _params(value), pattern_only=True)
        P.Initialize()
        st[value] = P.Stats()
    assert st[None]["a11_entry_bytes"] == st["Double"]["a11_entry_bytes"] == 8
    assert st["Single"]["a11_entry_bytes"] == 4
    for key in ("bytes_a11_level0", "bytes_a11_full_pass"):
        assert st[None][key] == st["Double"][key] > 0
        assert st["Single"][key] == st["Double"][key] / 2
    # the A11 term of bytes_apply (all levels) halves, nothing else changes: it is at least the level-0 saving
    saved = st["Double"]["bytes_apply"] - st["Single"]["bytes_apply"]
    assert saved >= st["Single"]["bytes_a11_level0"] and np.isfinite(saved)
