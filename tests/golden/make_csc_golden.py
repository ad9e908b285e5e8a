"""Generate tests/golden/csc_bridges.npz: the inputs and expected outputs of
test_gpu_parity.py::test_csc_bridges_vs_reference, so that the test needs
nothing outside the repository.

    python tests/golden/make_csc_golden.py

For every case of cases.CSC_CASES it stores
  <key>|p, <key>|i, <key>|x      the CSC input (cases.csc_fixture, seed 17)
  <key>|ep, <key>|ei, <key>|ex   the CSC of the SVT C_build_SVT_from_CSC()
                                 builds from it, as
                                 C_from_SVT_SparseMatrix_to_CsparseMatrix()
                                 returns it: zeros of @x dropped (NA and NaN
                                 are not zeros), 0-based rows in increasing
                                 order within each column
  <key>|col|<op>|<na_rm>, <key>|row|<op>|<na_rm>
                                 colStats / rowStats "sum" and "max" of that
                                 SVT, from the oracle's C restatement (which
                                 test_golden.py holds bit-for-bit to the
                                 reference's stored outputs)
When the reference's own C is built (oracle/_ref), every stored array is
checked against it byte for byte before the file is written.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
sys.path.insert(0, ROOT)
sys.path.insert(0, TESTS)

import cases  # noqa: E402
from oracle import port, refcall  # noqa: E402

OPS = ("sum", "max")


def canonical_csc(p, i, x, one_based):
    """(p, i, x) with zeros dropped and rows ordered within each column"""
    ep, ei, ex = [0], [], []
    for j in range(p.size - 1):
        rows = i[p[j]:p[j + 1]].astype(np.int64) - int(one_based)
        vals = x[p[j]:p[j + 1]]
        keep = vals != 0
        order = np.argsort(rows[keep], kind="stable")
        ei.append(rows[keep][order])
        ex.append(vals[keep][order])
        ep.append(ep[-1] + int(keep.sum()))
    return (np.array(ep, dtype=np.int32),
            np.concatenate(ei).astype(np.int32),
            np.concatenate(ex).astype(x.dtype))


def case_outputs(p, i, x, one_based):
    nrow, ncol = cases.CSC_DIM
    type_ = "double" if x.dtype == np.float64 else "integer"
    ep, ei, ex = canonical_csc(p, i, x, one_based)
    out = {"ep": ep, "ei": ei, "ex": ex}
    for op in OPS:
        for na_rm in (False, True):
            out["col|%s|%d" % (op, na_rm)] = port.colstats(
                nrow, ncol, ep, ei, ex, type_, op, na_rm)[0]
            out["row|%s|%d" % (op, na_rm)] = port.rowstats(
                nrow, ncol, ep, ei, ex, type_, op, na_rm)[0]
    return out


def reference_outputs(p, i, x, one_based):
    svt = refcall.build_SVT_from_CSC(cases.CSC_DIM, p.astype(np.int32), x, i,
                                     one_based)
    try:
        ep, ei, ex = refcall.from_SVT_to_CSC(svt)
        out = {"ep": ep, "ei": ei, "ex": ex}
        for op in OPS:
            for na_rm in (False, True):
                out["col|%s|%d" % (op, na_rm)] = refcall.colStats(
                    svt, op, na_rm=na_rm).value
                out["row|%s|%d" % (op, na_rm)] = refcall.rowStats(
                    svt, op, na_rm=na_rm).value
        return out
    finally:
        svt.release()


def main():
    nrow, ncol = cases.CSC_DIM
    out = {}
    for case in cases.CSC_CASES:
        key = cases.csc_key(*case)
        p, i, x = cases.csc_fixture(17, nrow, ncol, *case)
        res = case_outputs(p, i, x, case[1])
        if refcall.available():
            ref = reference_outputs(p, i, x, case[1])
            for k, v in res.items():
                r = np.asarray(ref[k])
                assert v.dtype == r.dtype and np.array_equal(
                    v.view(np.uint8), r.view(np.uint8)), (key, k)
        out.update({key + "|p": p, key + "|i": i, key + "|x": x})
        out.update({key + "|" + k: v for k, v in res.items()})
    path = os.path.join(HERE, "csc_bridges.npz")
    np.savez_compressed(path, **out)
    print("wrote %s: %d entries, %d bytes (%s)"
          % (path, len(out), os.path.getsize(path),
             "checked against oracle/_ref" if refcall.available()
             else "oracle/_ref not built: not checked against the reference"))


if __name__ == "__main__":
    main()
