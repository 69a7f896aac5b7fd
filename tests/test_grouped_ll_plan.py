"""CPU-only: the workspace formula and the host argument checks of the grouped likelihood with host-built covariance
functions (dense.ll_ws_doubles, dense.ll_workspace, cgp_large_ll_rows_dev)."""
import numpy as np


def test_ll_ws_doubles_matches_the_library():
    from cosmogp_b200 import build, dense, _lib
    build.build()
    L = _lib.lib()
    n = np.array([0, 1, 127, 128, 129, 600, 65535])
    got = dense.ll_ws_doubles(n)
    for i in range(len(n)):
        assert got[i] == L.cgp_large_ll_ws_doubles(int(n[i]))
    assert dense.ll_ws_doubles(300) == 384 * 384 + 2 * 384 + 6


def test_ll_workspace_is_capped(monkeypatch):
    """The workspace holds every object up to LL_WS_BYTES, and never less than the largest object."""
    import torch
    from cosmogp_b200 import dense
    made = []
    monkeypatch.setattr(torch, "empty", lambda n, **kw: made.append(n) or n)
    dense.ll_workspace([300, 60, 1000], "cpu")
    assert made[-1] == int(dense.ll_ws_doubles([300, 60, 1000]).sum())
    monkeypatch.setattr(dense, "LL_WS_BYTES", 8 * int(dense.ll_ws_doubles(1000)) + 8)
    dense.ll_workspace([1000, 1000, 60], "cpu")
    assert made[-1] == int(dense.ll_ws_doubles(1000)) + 1
    monkeypatch.setattr(dense, "LL_WS_BYTES", 8)
    dense.ll_workspace([1000, 2000], "cpu")
    assert made[-1] == int(dense.ll_ws_doubles(2000))


def test_entry_checks_before_any_launch():
    """NULL arguments, an unaligned or short workspace, a bad dim, an object id out of range and an oversized object
    are refused by the host checks, before any device work; no active object returns 0."""
    from cosmogp_b200 import build, _lib
    build.build()
    L = _lib.lib()
    fake = 1 << 20                                           # device pointers the checks never dereference
    hyp = np.array([1.0, 2.0, 1.0, 2.0])

    def call(n, work_doubles=1 << 40, dim=1, order=None, work=fake, hyp_rows=hyp, k=1):
        off = np.array([0, n], dtype=np.int64)
        o = None if order is None else np.asarray(order, dtype=np.int32)
        return L.cgp_large_ll_rows_dev(1, _lib.hptr(off), dim, fake, fake, None, None, _lib.hptr(hyp_rows), None, 0.05,
                                       0.0, 0, _lib.hptr(o), k, fake, fake, work, work_doubles, None)

    n0 = L.cgp_launch_count()
    assert call(65536) == -2 and "65535" in _lib.last_error()
    need = L.cgp_large_ll_ws_doubles(300)
    assert call(300, work_doubles=need - 1) == -2 and "workspace" in _lib.last_error()
    assert call(300, dim=3) == -1 and "dim" in _lib.last_error()
    assert call(300, order=[1]) == -1 and "object id" in _lib.last_error()
    assert call(300, work=fake + 8) == -1 and "aligned" in _lib.last_error()
    assert call(300, hyp_rows=None) == -1 and "NULL" in _lib.last_error()
    assert call(65536, dim=3, work=fake + 8) == -1 and "dim" in _lib.last_error()
    assert call(65536, hyp_rows=None, dim=3) == -1 and "NULL" in _lib.last_error()
    assert call(300, order=[], k=0) == 0
    assert L.cgp_launch_count() == n0
