"""ctypes loader for the C-ABI product library (include/lgu_corr.h -> liblgu_corr.so).

There is deliberately NO fallback: if the sm_100a library has not been built, importing the
ops fails loudly with the build command.  Nothing here imports oracle/.

Every entry point is bound with the argument and return types of its prototype (SIGNATURES), so a tensor address
cannot be cut to 32 bits, a Python float cannot reach a pointer, and `call` refuses a wrong argument count.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LGU_CORR_LIB") or os.path.join(_HERE, "liblgu_corr.so")   # override: kernel A/B experiments
ABI_VERSION = 1

_lib = None


class LguError(RuntimeError):
    """A C-ABI call returned a non-zero status (the reference raises RuntimeError via TORCH_CHECK)."""


class Ptr:
    """Argument type of every pointer parameter: None (NULL), an int address, anything with data_ptr() (a tensor), or a
    ctypes pointer, array or byref().  Anything else -- a float, say -- raises ctypes.ArgumentError."""

    _CTYPES = (ctypes._Pointer, ctypes.Array, type(ctypes.byref(ctypes.c_int())))

    @classmethod
    def from_param(cls, obj):
        if obj is None or isinstance(obj, int):
            return ctypes.c_void_p(obj)
        if hasattr(obj, "data_ptr"):
            return ctypes.c_void_p(obj.data_ptr())
        if isinstance(obj, cls._CTYPES):
            return obj
        raise TypeError(f"expected a pointer, got {type(obj).__name__}")


_P, _I, _LL, _F = (Ptr,), (ctypes.c_int,), (ctypes.c_longlong,), (ctypes.c_float,)

# (name, argument types[, return type]) for every prototype of include/lgu_corr.h, in header order.  An entry without a
# return type returns an int status (0 = LGU_OK).  tests/test_binding_cpu.py keeps this table and the header in step.
SIGNATURES = (
    ("lgu_abi_version", (), ctypes.c_int),
    ("lgu_build_info", (), ctypes.c_char_p),
    ("lgu_last_error_string", (), ctypes.c_char_p),
    ("lgu_corr_index_forward", _P * 3 + _I * 6 + _P),
    ("lgu_corr_index_backward", _P * 3 + _I * 6 + _P),
    ("lgu_defcorr_index_forward", _P * 4 + _I * 6 + _P),
    ("lgu_defcorr_index_backward", _P * 6 + _I * 6 + _P),
    ("lgu_gaussian_mask_forward", _P * 4 + _I * 6 + _P),
    ("lgu_gaussian_mask_backward", _P * 6 + _I * 6 + _P),
    ("lgu_lowmem_defsample_forward", _P * 5 + _I * 9 + _P),
    ("lgu_lowmem_workspace_bytes", _I * 8, ctypes.c_longlong),
    ("lgu_lowmem_defsample_forward_ws", _P * 5 + _I * 9 + _P + _LL + _P),
    ("lgu_altcorr_forward_ws", _P * 4 + _I * 8 + _P + _LL + _P),
    ("lgu_altcorr_forward", _P * 4 + _I * 8 + _P),
    ("lgu_build_pyramid", _P * 11 + _I * 8 + _P),
    ("lgu_corr_lookup_fused", _P * 9 + _I * 5 + _P),
    ("lgu_corr_lookup_fused_cum", _P * 11 + _I * 6 + _P),
    ("lgu_pack_conv1x1", _P * 2 + _I * 2 + _P),
    ("lgu_corr_lookup_fused_enc", _P * 12 + _I * 2 + _P * 2 + _I * 6 + _P),
    ("lgu_altcorr_lookup_fused", _P * 9 + _I * 7 + _P),
    ("lgu_altcorr_lookup_fused_into", _P * 9 + _I + _P + _I * 7 + _P),
    ("lgu_pack_conv1x1_f16", _P * 3 + _I * 2 + _P),
    ("lgu_altcorr_lookup_enc_into", _P * 12 + _I + _P + _I * 7 + _P),
    ("lgu_corr_lookup_fused_backward", _P * 14 + _I * 5 + _P),
    ("lgu_corr_lookup_fused_backward_accumulate", _P * 14 + _I * 5 + _P),
    ("lgu_corr_lookup_fused_backward_cum", _P * 15 + _I * 6 + _P),
    ("lgu_corr_lookup_fused_backward_win", _P * 17 + _I * 5 + _P),
    ("lgu_corr_lookup_fused_backward_gauss", _P * 21 + _I * 6 + _P),
    ("lgu_build_backward_gauss_window", _P * 8 + _I * 3 + _P),
    ("lgu_build_backward_gauss", _P * 11 + _I * 4 + _P),
    ("lgu_build_backward_fmaps", _P * 7 + _I * 5 + _P),
    ("lgu_tf32_split", _P + _F + _P * 2 + _LL + _P),
    ("lgu_build_pyramid_slots", _P * 12 + _I * 9 + _P),
    ("lgu_corr_lookup_fused_slots", _P * 10 + _I * 6 + _P),
    ("lgu_build_volume", _P * 7 + _I * 7 + _P),
    ("lgu_volume_half_mask", _P * 2 + _I * 4 + _P),
    ("lgu_build_volume_sparse", _P * 8 + _I * 7 + _P),
    ("lgu_build_boxes", _P * 7 + _I * 7 + _P),
    ("lgu_altcorr_lookup_boxes_into", _P * 10 + _I + _P + _I * 7 + _P),
    ("lgu_pack_fmaps", _P + _I + _P * 2 + _I * 3 + _P),
    ("lgu_offset_heads", _P * 5 + _I * 4 + _F + _P),
    ("lgu_peer_alloc", _LL + _P * 2),
    ("lgu_peer_open", _P * 2),
    ("lgu_peer_close", _P),
    ("lgu_peer_free", _P),
)
_RETURNS_STATUS = {name for name, _, *ret in SIGNATURES if not ret}


def build(verbose=False):
    """Compile liblgu_corr.so in-tree with nvcc for sm_100a (seconds; no GPU needed)."""
    import subprocess
    cmd = ["make", "-C", os.path.join(_HERE, "csrc"), "-j8"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout[-4000:], res.stderr[-4000:])
    if res.returncode != 0:
        raise RuntimeError("building liblgu_corr.so failed (see output above)")
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: the sm_100a CUDA library has not been built. "
                "Run `python -c 'import __graft_entry__ as g; g.build()'` (or `make -C lgu-slam_b200/csrc`). "
                "There is no CPU fallback.")
        L = ctypes.CDLL(LIB_PATH)
        for name, argtypes, *ret in SIGNATURES:
            fn = getattr(L, name)
            fn.argtypes = argtypes
            fn.restype = ret[0] if ret else ctypes.c_int
        got = L.lgu_abi_version()
        if got != ABI_VERSION:
            raise ImportError(f"liblgu_corr.so ABI version {got} != expected {ABI_VERSION}; rebuild it")
        _lib = L
    return _lib


LAUNCHES = 0          # C-ABI calls that returned a status so far (each launches at least one kernel, except lgu_peer_*)


def check(status, what):
    global LAUNCHES
    LAUNCHES += 1
    if status != 0:
        msg = lib().lgu_last_error_string().decode("utf-8", "replace")
        raise LguError(f"{what} failed (status {status}): {msg}")


def pointer_array(tensors):
    """A host array of device pointers for the `T* const*` parameters (lgu_build_backward_fmaps); None entries are NULL."""
    return (ctypes.c_void_p * len(tensors))(*[None if t is None else t.data_ptr() for t in tensors])


def call(name, *args):
    """Call entry point `name` with exactly its declared arguments; a non-zero status raises LguError.  Returns what the
    function returns (the status, or the value of an entry point that returns no status)."""
    fn = getattr(lib(), name)
    if len(args) != len(fn.argtypes):
        raise TypeError(f"{name} takes {len(fn.argtypes)} arguments, got {len(args)}")
    res = fn(*args)
    if name in _RETURNS_STATUS:
        check(res, name)
    return res
