"""CPU-only: the chunk planner and the host helpers of the grouped predictive covariance (dense.plan_chunks,
dense.cov_ws_doubles, dense._gather)."""
import numpy as np


def test_plan_chunks_output_budget():
    from cosmogp_b200 import dense
    out = np.full(8000, 8 * 100 * 100)                       # 80 kB matrices: chunks of 3 355 objects in 256 MB
    b = dense.plan_chunks(out)
    assert b == [0, 3355, 6710, 8000]


def test_plan_chunks_both_budgets():
    from cosmogp_b200 import dense
    assert dense.plan_chunks([1, 2, 3], [5, 5, 5], out_budget=3, ws_budget=100) == [0, 2, 3]
    assert dense.plan_chunks([1, 1, 1, 1], [40, 40, 40, 40], out_budget=100, ws_budget=100) == [0, 2, 4]
    assert dense.plan_chunks([500, 1, 1], [1, 1, 1], out_budget=100, ws_budget=100) == [0, 1, 3]   # oversize alone
    assert dense.plan_chunks([0, 0], [0, 0]) == [0, 2]
    assert dense.plan_chunks([]) == [0, 0]


def test_cov_ws_doubles_matches_the_library():
    from cosmogp_b200 import build, dense, _lib
    build.build()
    L = _lib.lib()
    n = np.array([0, 1, 127, 128, 129, 600, 65535])
    m = np.array([0, 1000, 1, 7, 300, 129, 2])
    got = dense.cov_ws_doubles(n, m)
    for i in range(len(n)):
        assert got[i] == L.cgp_large_cov_ws_doubles(int(n[i]), int(m[i]))
    assert dense.cov_ws_doubles(300, 100) == 384 * 384 + 128 * 384 + 128 * 128


def test_gather_csr():
    from cosmogp_b200 import dense
    flat = np.arange(20.0).reshape(10, 2)
    off = np.array([0, 3, 3, 7, 10])
    rows, new_off = dense._gather(flat, off, np.array([2, 1, 0]))
    np.testing.assert_array_equal(new_off, [0, 4, 4, 7])
    np.testing.assert_array_equal(rows, np.concatenate([flat[3:7], flat[0:3]]))


def test_entry_size_limits_refused_before_any_launch():
    """Objects and grids are limited to 65408 points (padded to 128, at most the 65535 rows an auto-covariance build
    takes); larger ones, and a too small workspace, are refused by the host checks, before any device work."""
    from cosmogp_b200 import build, _lib
    build.build()
    L = _lib.lib()
    fake = 1 << 20                                           # device pointers the checks never dereference
    hyp, nug = np.array([1.0, 2.0]), np.array([0.05])
    info = fake

    def call(n, m_shared=None, goff=None, m=0, work_doubles=1 << 40):
        off = np.array([0, n], dtype=np.int64)
        coff = np.array([0, m * m], dtype=np.int64)
        return L.cgp_large_covariance_dev(1, _lib.hptr(off), 1, fake, None, _lib.hptr(hyp), _lib.hptr(nug), 0.0, 0.0, 0,
                                          fake, _lib.hptr(goff), 0 if m_shared is None else m_shared, None, 1, fake,
                                          _lib.hptr(coff), info, fake, work_doubles, None)

    assert call(65409) == -2 and "65408" in _lib.last_error()
    assert call(10, m_shared=65409, m=65409) == -2 and "65408" in _lib.last_error()
    assert call(10, goff=np.array([0, 65409], dtype=np.int64), m=65409) == -2 and "65408" in _lib.last_error()
    assert call(65408, m_shared=65408, m=65408, work_doubles=1) == -2 and "workspace" in _lib.last_error()
    assert call(10, m_shared=7, m=6) == -1 and "coff" in _lib.last_error()
