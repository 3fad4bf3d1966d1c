"""Argument checks of the backend encoder entry points (lgu_pack_conv1x1_f16, lgu_altcorr_lookup_enc_into): bad pointers
and sizes are refused with an error code before any device work, so these calls run without a GPU."""
import ctypes
import os

import pytest

LGU_OK, LGU_ERR_BAD_ARG, LGU_ERR_UNSUPPORTED = 0, 1, 3


@pytest.fixture(scope="module")
def lib():
    import lgu_slam_b200
    if not os.path.exists(lgu_slam_b200._lib.LIB_PATH):
        lgu_slam_b200._lib.build()
    L = ctypes.CDLL(lgu_slam_b200._lib.LIB_PATH)
    L.lgu_last_error_string.restype = ctypes.c_char_p
    return L


A = ctypes.c_void_p(1 << 20)           # a 16-byte aligned address that is never dereferenced


def _pack(L, weight=A, bias=A, packed=A, oc=128, ic=196):
    return L.lgu_pack_conv1x1_f16(weight, bias, packed, oc, ic, None)


def _lookup(L, boxes0=A, boxes1=None, lvl0=None, lvl1=A, packed=A, enc=A, E=2, H=48, W=64, levels=4, radius=3,
            shared_offsets=1, apply_mask=0):
    return L.lgu_altcorr_lookup_enc_into(boxes0, boxes1, lvl0, lvl1, A, A, A, A, A, packed, enc, None, 1, None, E, H, W,
                                         levels, radius, shared_offsets, apply_mask, None)


def test_pack_refuses_null_misaligned_and_other_shapes(lib):
    assert _pack(lib, weight=None) == LGU_ERR_BAD_ARG and b"null" in lib.lgu_last_error_string()
    assert _pack(lib, packed=None) == LGU_ERR_BAD_ARG
    assert _pack(lib, packed=ctypes.c_void_p((1 << 20) + 8)) == LGU_ERR_BAD_ARG
    assert b"aligned" in lib.lgu_last_error_string()
    for oc, ic in ((64, 196), (128, 128), (196, 128)):
        assert _pack(lib, oc=oc, ic=ic) == LGU_ERR_BAD_ARG
        assert b"196 -> 128" in lib.lgu_last_error_string()


def test_lookup_refuses_null_and_misaligned_pointers(lib):
    assert _lookup(lib, packed=None) == LGU_ERR_BAD_ARG and b"null" in lib.lgu_last_error_string()
    assert _lookup(lib, enc=None) == LGU_ERR_BAD_ARG
    assert _lookup(lib, boxes0=None, lvl0=None) == LGU_ERR_BAD_ARG                # level 0: neither boxes nor a volume
    assert _lookup(lib, lvl1=None) == LGU_ERR_BAD_ARG                             # level 1: neither boxes nor a volume
    assert _lookup(lib, packed=ctypes.c_void_p((1 << 20) + 8)) == LGU_ERR_BAD_ARG
    assert b"aligned" in lib.lgu_last_error_string()
    assert _lookup(lib, enc=ctypes.c_void_p((1 << 20) + 4)) == LGU_ERR_BAD_ARG
    assert _lookup(lib, boxes0=ctypes.c_void_p((1 << 20) + 4)) == LGU_ERR_BAD_ARG
    assert _lookup(lib, boxes1=A, boxes0=None, lvl0=A) == LGU_ERR_BAD_ARG         # compact level 1 needs compact level 0


def test_lookup_refuses_bad_sizes_and_reports_unsupported_grids(lib):
    assert _lookup(lib, E=-1) == LGU_ERR_BAD_ARG
    assert _lookup(lib, H=0) == LGU_ERR_BAD_ARG and b"bad sizes" in lib.lgu_last_error_string()
    assert _lookup(lib, W=-64) == LGU_ERR_BAD_ARG
    for kw in (dict(W=48), dict(H=44), dict(levels=3), dict(radius=2)):
        assert _lookup(lib, **kw) == LGU_ERR_UNSUPPORTED, kw
    assert _lookup(lib, E=0) == LGU_OK                                           # an empty edge set is a no-op
