"""CPU-only: the workspace formula and the host argument checks of the grouped large-object leave-one-out
(dense.loo_ws_doubles, cgp_large_loo_objhyp_dev)."""
import numpy as np


def test_loo_ws_doubles_matches_the_library():
    from cosmogp_b200 import build, dense, _lib
    build.build()
    L = _lib.lib()
    n = np.array([0, 1, 127, 128, 129, 300, 1000, 20000, 65408])
    for chunk in (128, 384, 1024, 20096, 1 << 20):
        got = dense.loo_ws_doubles(n, chunk)
        for i in range(len(n)):
            assert got[i] == L.cgp_large_loo_ws_doubles(int(n[i]), chunk)
    assert dense.loo_ws_doubles(300, 128) == 384 * 384 + 128 * 384 + 7 * 384 + 2
    assert dense.loo_ws_doubles(300, 1024) == 2 * 384 * 384 + 7 * 384 + 2
    assert dense.loo_chunk_rows(384) == 384 and dense.loo_chunk_rows(1024, 300) == 256
    assert dense.loo_chunk_rows(20096) == 20096 and dense.loo_chunk_rows(65408) == (4 << 30) // (8 * 65408) // 128 * 128


def test_entry_checks_before_any_launch():
    """A bad mode, a chunk_rows that is not a positive multiple of 128, an oversized object and a short workspace are
    refused by the host checks, before any device work; no active object launches nothing, but a bad mode or chunk_rows
    is refused even then, after a negative object count."""
    from cosmogp_b200 import build, _lib
    build.build()
    L = _lib.lib()
    fake = 1 << 20                                           # device pointers the checks never dereference
    hyp = np.array([1.0, 2.0])

    def call(n, mode=_lib.CGP_LOO_PLAIN, chunk_rows=128, work_doubles=1 << 40, n_active=1):
        off = np.array([0, n], dtype=np.int64)
        order = np.zeros(1, dtype=np.int32)
        return L.cgp_large_loo_objhyp_dev(1, _lib.hptr(off), 1, fake, fake, None, None, _lib.hptr(hyp), None, 0.05, 0.0, 0,
                                          mode, _lib.hptr(order), n_active, fake, fake, fake, fake, fake, chunk_rows, fake,
                                          work_doubles, None)

    n0 = L.cgp_launch_count()
    assert call(300, mode=2) == -1 and "mode" in _lib.last_error()
    assert call(300, chunk_rows=100) == -1 and "chunk_rows" in _lib.last_error()
    assert call(300, chunk_rows=0) == -1 and "chunk_rows" in _lib.last_error()
    assert call(65409) == -2 and "65408" in _lib.last_error()
    need = L.cgp_large_loo_ws_doubles(300, 128)
    assert call(300, work_doubles=need - 1) == -2 and "workspace" in _lib.last_error()
    assert L.cgp_large_loo_ws_doubles(300, 0) == 0 and L.cgp_large_loo_ws_doubles(-1, 128) == 0
    assert call(300, n_active=0) == 0
    assert call(300, mode=2, n_active=0) == -1 and "mode" in _lib.last_error()
    assert call(300, chunk_rows=100, n_active=0) == -1 and "chunk_rows" in _lib.last_error()
    assert call(300, mode=2, n_active=-1) == -1 and "negative" in _lib.last_error()
    assert L.cgp_launch_count() == n0
