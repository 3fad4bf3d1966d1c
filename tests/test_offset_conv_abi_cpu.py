"""Argument checks of the conv3x3 entry points (the offset heads' convolutions): null pointers, a misaligned workspace and
unsupported sizes are refused with LGU_ERR_BAD_ARG and a message naming the argument before any device work, and an
empty edge set is a no-op, so these calls run without a GPU."""
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
    L.lgu_conv3x3_workspace_bytes.restype = ctypes.c_longlong
    return L


A = ctypes.c_void_p(1 << 20)           # a 256-byte aligned address that is never dereferenced
WS = ctypes.c_longlong(1 << 40)
SIZES = dict(E=2, C_in=256, C_out=98, H=48, W=64)


def _sizes(kw):
    s = dict(SIZES, **kw)
    return s["E"], s["C_in"], s["C_out"], s["H"], s["W"]


def _pack(L, x=A, hi=A, lo=A, **kw):
    E, C_in, _, H, W = _sizes(kw)
    return L.lgu_conv3x3_pack(x, hi, lo, E, C_in, H, W, None)


def _fwd(L, x_hi=A, x_lo=A, weight=A, bias=A, y=A, workspace=A, ws=WS, **kw):
    return L.lgu_conv3x3_forward(x_hi, x_lo, weight, bias, y, workspace, ws, *_sizes(kw), None)


def _bwd_in(L, gy_hi=A, gy_lo=A, weight=A, g_x=A, workspace=A, ws=WS, **kw):
    return L.lgu_conv3x3_backward_input(gy_hi, gy_lo, weight, g_x, workspace, ws, *_sizes(kw), None)


def _bwd_w(L, x_hi=A, x_lo=A, g_y=A, g_w=A, g_b=A, workspace=A, ws=WS, **kw):
    return L.lgu_conv3x3_backward_weight(x_hi, x_lo, g_y, g_w, g_b, workspace, ws, *_sizes(kw), None)


CALLS = {"pack": (_pack, ["x", "hi", "lo"]),
         "forward": (_fwd, ["x_hi", "x_lo", "weight", "y", "workspace"]),
         "backward_input": (_bwd_in, ["gy_hi", "gy_lo", "weight", "g_x", "workspace"]),
         "backward_weight": (_bwd_w, ["x_hi", "x_lo", "g_y", "workspace"])}      # g_w, g_b: either may be NULL


@pytest.mark.parametrize("op, arg", [(op, a) for op, (_, args) in CALLS.items() for a in args])
def test_refuses_a_null_required_pointer(lib, op, arg):
    fn, _ = CALLS[op]
    assert fn(lib, **{arg: None}) == LGU_ERR_BAD_ARG
    assert f"{arg} is NULL".encode() in lib.lgu_last_error_string()


def test_backward_weight_refuses_no_output_and_takes_a_missing_one(lib):
    assert _bwd_w(lib, g_w=None, g_b=None) == LGU_ERR_BAD_ARG
    assert b"g_w and g_b are both NULL" in lib.lgu_last_error_string()
    # without g_w, only g_y and g_b are read: the planes and the workspace may be NULL; E = 0 never launches
    assert _bwd_w(lib, g_w=None, x_hi=None, x_lo=None, workspace=None, E=0) == LGU_OK
    assert _bwd_w(lib, g_w=None, x_hi=None, x_lo=None, workspace=None, g_y=None) == LGU_ERR_BAD_ARG
    assert b"g_y is NULL" in lib.lgu_last_error_string()


@pytest.mark.parametrize("op", ["forward", "backward_input", "backward_weight"])
def test_refuses_a_misaligned_or_short_workspace(lib, op):
    fn, _ = CALLS[op]
    assert fn(lib, workspace=ctypes.c_void_p((1 << 20) + 16)) == LGU_ERR_BAD_ARG
    assert b"workspace is not 256-byte aligned" in lib.lgu_last_error_string()
    assert fn(lib, ws=ctypes.c_longlong(1024)) == LGU_ERR_BAD_ARG
    assert b"workspace_bytes=1024" in lib.lgu_last_error_string()


def test_refuses_misaligned_planes(lib):
    assert _fwd(lib, x_lo=ctypes.c_void_p((1 << 20) + 4)) == LGU_ERR_BAD_ARG
    assert b"x_lo is not 16-byte aligned" in lib.lgu_last_error_string()


@pytest.mark.parametrize("kw, word", [(dict(C_out=0), b"C_out=0"), (dict(C_out=129), b"C_out=129"),
                                      (dict(C_in=100), b"C_in=100"), (dict(C_in=0), b"C_in=0"),
                                      (dict(W=48), b"W=48"), (dict(W=96), b"W=96"), (dict(W=0), b"W=0"),
                                      (dict(H=3, W=32), b"H=3"), (dict(E=-1), b"E=-1")])
@pytest.mark.parametrize("op", ["forward", "backward_input", "backward_weight"])
def test_refuses_unsupported_sizes(lib, op, kw, word):
    fn, _ = CALLS[op]
    assert fn(lib, **kw) == LGU_ERR_BAD_ARG
    msg = lib.lgu_last_error_string()
    assert b"bad size" in msg and word in msg, msg
    assert lib.lgu_conv3x3_workspace_bytes(*_sizes(kw)) == -1


@pytest.mark.parametrize("kw, word", [(dict(W=48), b"W=48"), (dict(H=3, W=32), b"H=3"), (dict(E=-1), b"E=-1")])
def test_pack_refuses_unsupported_sizes(lib, kw, word):
    assert _pack(lib, **kw) == LGU_ERR_BAD_ARG
    assert word in lib.lgu_last_error_string()


def test_empty_edge_sets_are_a_no_op(lib):
    for op, (fn, args) in CALLS.items():
        assert fn(lib, E=0) == LGU_OK, op
        assert fn(lib, E=0, **{a: None for a in args}) == LGU_OK, op


def test_workspace_size_covers_both_grids(lib):
    for H, W in ((48, 64), (24, 32)):
        for E in (1, 96):
            n = lib.lgu_conv3x3_workspace_bytes(E, 256, 98, H, W)
            # the weight gradient's split g_y planes [E, 112, H*W] x 2 are the largest part
            assert n >= 2 * E * 112 * H * W * 4, (E, H, W, n)
