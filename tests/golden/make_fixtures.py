"""Regenerates tests/golden/*.npz from the reference's shipped MatrixMarket fixtures.

    python tests/golden/make_fixtures.py <checkout of nlesc-smcm/hymls>

Sources: testSuite/data/DrivenCavity/{32x32,64x64}/Re0, 32x32/Re1000, 16x16x16/Re0
(jac.mtx / rhs.mtx / sol.mtx), stored losslessly (float64) in CSR form.
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", ".."))
from oracle import galeri  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def dump(ref, name, sub, with_vec=True):
    src = os.path.join(ref, "testSuite", "data", "DrivenCavity", sub)
    A = galeri.read_mtx(os.path.join(src, "jac.mtx"))
    out = dict(indptr=A.indptr.astype(np.int32), indices=A.indices.astype(np.int32), data=A.data,
               shape=np.asarray(A.shape))
    if with_vec:
        out["rhs"] = galeri.read_mtx(os.path.join(src, "rhs.mtx"))
        out["sol"] = galeri.read_mtx(os.path.join(src, "sol.mtx"))
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    dump(sys.argv[1], "cavity2d_32_Re0", "32x32/Re0")
    dump(sys.argv[1], "cavity2d_64_Re0", "64x64/Re0")
    dump(sys.argv[1], "cavity2d_32_Re1000", "32x32/Re1000")
    dump(sys.argv[1], "cavity3d_16_Re0", "16x16x16/Re0")
