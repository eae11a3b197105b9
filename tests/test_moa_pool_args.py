"""ssd_moa_create_pool validates its arguments before it touches a device: these checks need no GPU."""
import ctypes as C

import numpy as np


def test_create_pool_argument_errors_need_no_gpu():
    from sequential_social_dilemma_games_b200 import _lib
    L = _lib.lib
    big = np.zeros(4 * ((32 + 17 * 15) * 512 + 128 * 512 + 512 + 128 * 64 + 64), np.float32)
    bp = big.ctypes.data_as(C.c_void_p)
    out = C.c_void_p()
    for K in (0, 256, -1):
        assert L.ssd_moa_create_pool(0, K, 5, 8, bp, bp, bp, bp, bp, C.byref(out)) == -1 and not out.value, K
        assert b"1..255" in L.ssd_last_error()
    for n, a in ((1, 8), (17, 2), (5, 0), (5, 16), (9, 9)):   # N, A and (N - 1) A as ssd_moa_create
        assert L.ssd_moa_create_pool(0, 3, n, a, bp, bp, bp, bp, bp, C.byref(out)) == -1 and not out.value, (n, a)
    for k in range(5):
        ptrs = [bp] * 5
        ptrs[k] = None
        assert L.ssd_moa_create_pool(0, 3, 5, 8, *ptrs, C.byref(out)) == -1 and not out.value, k
        assert b"null" in L.ssd_last_error()
    assert L.ssd_moa_create_pool(0, 3, 5, 8, bp, bp, bp, bp, bp, None) == -1 and b"null" in L.ssd_last_error()
    # the plain MOA still takes 1 or N weight sets only
    assert L.ssd_moa_create(0, 3, 5, 8, bp, bp, bp, bp, bp, C.byref(out)) == -1 and not out.value


def test_pool_step_rejects_null_arguments_without_gpu():
    from sequential_social_dilemma_games_b200 import _lib
    L = _lib.lib
    args = [C.c_void_p(16)] * 12
    assert L.ssd_moa_pool_step(None, *args, 5, 0, 1.0, None) == -1 and b"bad argument" in L.ssd_last_error()
    assert L.ssd_moa_pool_step(C.c_void_p(16), args[0], None, *args[2:], 5, 0, 1.0, None) == -1   # policy_ids
    assert b"bad argument" in L.ssd_last_error()
