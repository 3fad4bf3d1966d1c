"""Argument checks of lgu_offset_heads_backward: null pointers and unsupported sizes are refused with LGU_ERR_BAD_ARG
and a message naming the argument before any device work, and an empty edge set is a no-op, so these calls run without
a GPU."""
import ctypes
import os

import pytest

LGU_OK, LGU_ERR_BAD_ARG = 0, 1


@pytest.fixture(scope="module")
def lib():
    import lgu_slam_b200
    if not os.path.exists(lgu_slam_b200._lib.LIB_PATH):
        lgu_slam_b200._lib.build()
    L = ctypes.CDLL(lgu_slam_b200._lib.LIB_PATH)
    L.lgu_last_error_string.restype = ctypes.c_char_p
    return L


A = ctypes.c_void_p(1 << 20)           # a 16-byte aligned address that is never dereferenced


def _bwd(L, c0=A, c1=A, stats=A, g0=A, g1=A, g_c0=A, g_c1=A, scratch=A, E=2, CH=98, H=48, W=64):
    return L.lgu_offset_heads_backward(c0, c1, stats, g0, g1, g_c0, g_c1, scratch, E, CH, H, W, None)


@pytest.mark.parametrize("arg", ["c0", "c1", "stats", "g_c0", "g_c1", "scratch"])
def test_backward_refuses_a_null_required_pointer(lib, arg):
    assert _bwd(lib, **{arg: None}) == LGU_ERR_BAD_ARG
    assert f"{arg} is NULL".encode() in lib.lgu_last_error_string()


def test_backward_refuses_misaligned_scratch(lib):
    assert _bwd(lib, scratch=ctypes.c_void_p((1 << 20) + 4)) == LGU_ERR_BAD_ARG
    assert b"scratch is not 8-byte aligned" in lib.lgu_last_error_string()


@pytest.mark.parametrize("kw, word", [(dict(W=48), b"W=48"), (dict(W=0), b"W=0"), (dict(H=47), b"H=47"),
                                      (dict(H=0), b"H=0"), (dict(CH=129), b"CH=129"), (dict(CH=0), b"CH=0"),
                                      (dict(E=-1), b"E=-1")])
def test_backward_refuses_unsupported_sizes(lib, kw, word):
    assert _bwd(lib, **kw) == LGU_ERR_BAD_ARG
    msg = lib.lgu_last_error_string()
    assert b"bad size" in msg and word in msg, msg


def test_backward_takes_missing_upstream_gradients_and_empty_edge_sets(lib):
    # G0 / G1 may be NULL (zero gradients): with bad sizes the call still fails on the sizes, not on them
    assert _bwd(lib, g0=None, g1=None, W=48) == LGU_ERR_BAD_ARG
    assert b"W=48" in lib.lgu_last_error_string()
    assert _bwd(lib, E=0) == LGU_OK
    assert _bwd(lib, E=0, c0=None, c1=None, stats=None, g_c0=None, g_c1=None, scratch=None) == LGU_OK
