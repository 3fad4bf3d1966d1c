"""The typed binding of the C ABI (lgu-slam_b200/_lib.py) against include/lgu_corr.h, without a GPU: the signature table
declares every prototype with the header's argument kinds, lib() applies it, every call the package makes names a
declared entry point with the declared number of arguments, and a wrong argument fails loudly instead of being
passed through as a truncated or shifted value."""
import ast
import ctypes
import glob
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "lgu-slam_b200")


@pytest.fixture(scope="module")
def binding():
    import lgu_slam_b200
    if not os.path.exists(lgu_slam_b200._lib.LIB_PATH):
        lgu_slam_b200._lib.build()
    return lgu_slam_b200._lib


def _kind(decl):
    """'const float* coords' -> 'pointer'; 'long long bytes' -> 'long long'; 'int E' -> 'int'; 'float eps' -> 'float'."""
    if "*" in decl:
        return "pointer"
    words = decl.split()[:-1]                   # drop the parameter name
    return " ".join(w for w in words if w != "const")


def _prototypes():
    """[(name, return kind, [argument kinds])] of include/lgu_corr.h, in header order."""
    hdr = open(os.path.join(ROOT, "include", "lgu_corr.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    out = []
    for ret, name, args in re.findall(r"LGU_API[ \t]+([^\n;(]*?)\s*\b(lgu_\w+)\s*\(([^)]*)\)\s*;", hdr):
        args = " ".join(args.split())
        kinds = [] if args in ("", "void") else [_kind(a) for a in args.split(",")]
        out.append((name, "pointer" if "*" in ret else ret.strip(), kinds))
    return out


def _table():
    import lgu_slam_b200
    return lgu_slam_b200._lib


def _ctype_kind(t):
    return {_table().Ptr: "pointer", ctypes.c_char_p: "pointer", ctypes.c_int: "int", ctypes.c_longlong: "long long",
            ctypes.c_float: "float"}.get(t, repr(t))


def test_signature_table_matches_the_header():
    protos = _prototypes()
    assert len(protos) == 45
    table = _table().SIGNATURES
    assert [s[0] for s in table] == [p[0] for p in protos], "one entry per prototype, in header order"
    for (name, ret, kinds), (_, argtypes, *rt) in zip(protos, table):
        assert [_ctype_kind(t) for t in argtypes] == kinds, name
        assert _ctype_kind(rt[0] if rt else ctypes.c_int) == ret, name


def test_lib_binds_every_entry_point(binding):
    L = binding.lib()
    for name, argtypes, *rt in binding.SIGNATURES:
        fn = getattr(L, name)
        assert tuple(fn.argtypes) == tuple(argtypes), name
        assert fn.restype is (rt[0] if rt else ctypes.c_int), name
    assert L.lgu_lowmem_workspace_bytes.restype is ctypes.c_longlong


def _calls():
    """Every _launch(...) / _lib.call(...) in the package's Python: (file, line, [candidate names], argument count);
    an entry whose names or count cannot be read statically has names None."""
    found = []
    for path in sorted(glob.glob(os.path.join(PKG, "**", "*.py"), recursive=True)):
        tree = ast.parse(open(path).read(), path)
        skip = set()
        for fn in ast.walk(tree):                # the forwarding body of _launch itself
            if isinstance(fn, ast.FunctionDef) and fn.name == "_launch":
                skip.update(id(n) for n in ast.walk(fn))
        for node in ast.walk(tree):
            if not isinstance(node, ast.Call) or id(node) in skip:
                continue
            f = node.func
            if isinstance(f, ast.Name) and f.id == "_launch":
                fixed, extra = 2, 1                # name, device ... + the stream _launch appends
            elif isinstance(f, ast.Attribute) and f.attr == "call" and isinstance(f.value, ast.Name) and f.value.id == "_lib":
                fixed, extra = 1, 0
            else:
                continue
            where = (os.path.relpath(path, ROOT), node.lineno)
            first = node.args[0] if node.args else None
            if isinstance(first, ast.IfExp):
                names = [first.body, first.orelse]
            else:
                names = [first]
            if node.keywords or any(isinstance(a, ast.Starred) for a in node.args) or \
                    not all(isinstance(n, ast.Constant) and isinstance(n.value, str) for n in names):
                found.append(where + (None, None))
                continue
            found.append(where + ([n.value for n in names], len(node.args) - fixed + extra))
    return found


def test_every_call_site_names_a_declared_entry_point_with_its_argument_count():
    declared = {name: len(argtypes) for name, argtypes, *_ in _table().SIGNATURES}
    calls = _calls()
    assert len(calls) >= 40, "the scan must see the operator layer's calls"
    for path, line, names, count in calls:
        assert names is not None, f"{path}:{line}: call not countable (starred / keyword arguments or a computed name)"
        for name in names:
            assert name in declared, f"{path}:{line}: {name} is not in the signature table"
            assert count == declared[name], f"{path}:{line}: {name} takes {declared[name]} arguments, {count} passed"
    for path in glob.glob(os.path.join(PKG, "**", "*.py"), recursive=True):
        if not path.endswith("_lib.py"):
            assert "_lib.lib()" not in open(path).read(), f"{path} bypasses the typed binding"


def test_call_checks_the_status(binding):
    n0 = binding.LAUNCHES
    with pytest.raises(binding.LguError, match=r"status 1\).*null"):
        binding.call("lgu_corr_index_forward", None, None, None, 1, 4, 4, 4, 4, 1, None)
    assert binding.LAUNCHES == n0 + 1
    assert binding.call("lgu_corr_index_forward", 16, 16, 16, 0, 4, 4, 4, 4, 1, None) == 0    # empty edge set: no-op
    assert binding.call("lgu_lowmem_workspace_bytes", 1, 2, 48, 64, 48, 64, 128, 3) == 0      # N != 1: not covered
    assert binding.call("lgu_lowmem_workspace_bytes", 2048, 1, 48, 64, 48, 64, 128, 3) > 1 << 32   # long long, whole
    assert binding.LAUNCHES == n0 + 2                        # size queries are no launches


def test_call_refuses_wrong_arguments(binding):
    with pytest.raises(TypeError, match="takes 10 arguments, got 11"):
        binding.call("lgu_corr_index_forward", None, None, None, 0, 4, 4, 4, 4, 1, None, None)
    with pytest.raises(TypeError, match="takes 10 arguments, got 9"):
        binding.call("lgu_corr_index_forward", None, None, None, 0, 4, 4, 4, 4, 1)
    with pytest.raises(ctypes.ArgumentError):
        binding.call("lgu_corr_index_forward", 1.5, None, None, 0, 4, 4, 4, 4, 1, None)
    with pytest.raises(ctypes.ArgumentError):
        binding.call("lgu_corr_index_forward", None, None, None, 0.0, 4, 4, 4, 4, 1, None)


def test_pointer_type_accepts_addresses_tensors_and_ctypes_references(binding):
    import torch
    P = binding.Ptr
    t = torch.zeros(4)
    buf = ctypes.create_string_buffer(64)
    assert P.from_param(None).value is None
    assert P.from_param(1 << 40).value == 1 << 40                     # no truncation to 32 bits
    assert P.from_param(t).value == t.data_ptr()
    for ref in (buf, ctypes.byref(ctypes.c_void_p()), ctypes.pointer(ctypes.c_int())):
        assert P.from_param(ref) is ref
    for bad in (1.5, "ptr", b"ptr", [t]):
        with pytest.raises(TypeError):
            P.from_param(bad)
