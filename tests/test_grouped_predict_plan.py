"""CPU-only: the workspace formula and the host argument checks of the grouped large-object prediction
(dense.pred_ws_doubles, cgp_large_predict_objhyp_dev)."""
import numpy as np


def test_pred_ws_doubles_matches_the_library():
    from cosmogp_b200 import build, dense, _lib
    build.build()
    L = _lib.lib()
    n = np.array([0, 1, 127, 128, 129, 600, 65408])
    rows = np.array([0, 1000, 1, 0, 300, 129, 2])
    got = dense.pred_ws_doubles(n, rows)
    for i in range(len(n)):
        assert got[i] == L.cgp_large_pred_ws_doubles(int(n[i]), int(rows[i]))
    assert dense.pred_ws_doubles(300, 100) == 384 * 384 + 3 * 384 + 128 * 384
    assert dense.pred_ws_doubles(300, 0) == 384 * 384 + 3 * 384


def test_entry_checks_before_any_launch():
    """Oversized objects, a grid CSR that disagrees with the output CSR, a bad chunk_rows and a short workspace are
    refused by the host checks, before any device work.  A bad chunk_rows is checked after the alignment of the
    workspace and before its size, and not at all without an active object."""
    from cosmogp_b200 import build, _lib
    build.build()
    L = _lib.lib()
    fake = 1 << 20                                           # device pointers the checks never dereference
    hyp = np.array([1.0, 2.0])

    def call(n, m=10, moff_m=None, chunk_rows=128, work_doubles=1 << 40, var=fake, k=1, work=fake):
        off = np.array([0, n], dtype=np.int64)
        moff = np.array([0, m if moff_m is None else moff_m], dtype=np.int64)
        return L.cgp_large_predict_objhyp_dev(k, _lib.hptr(off), 1, fake, fake, None, None, _lib.hptr(hyp), None, 0.05,
                                              0.0, 0, fake, None, m, None, None, 1, _lib.hptr(moff), fake, var, fake,
                                              chunk_rows, work, work_doubles, None)

    n0 = L.cgp_launch_count()
    assert call(65409) == -2 and "65408" in _lib.last_error()
    assert call(300, moff_m=11) == -1 and "moff" in _lib.last_error()
    assert call(300, chunk_rows=100) == -1 and "chunk_rows" in _lib.last_error()
    need = L.cgp_large_pred_ws_doubles(300, 10)
    assert call(300, work_doubles=need - 1) == -2 and "workspace" in _lib.last_error()
    assert call(300, m=0, moff_m=0, work_doubles=L.cgp_large_pred_ws_doubles(300, 0) - 1, var=None) == -2
    assert call(300, chunk_rows=100, work=fake + 8) == -1 and "aligned" in _lib.last_error()
    assert call(300, chunk_rows=100, work_doubles=1) == -1 and "chunk_rows" in _lib.last_error()
    assert call(300, chunk_rows=100, k=0) == 0
    assert L.cgp_launch_count() == n0
