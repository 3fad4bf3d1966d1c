"""The typed binding of include/lgu_corr_ext.h (the entry points added after the version-1 set of lgu_corr.h) without a
GPU: EXT_SIGNATURES declares every prototype of that header with its argument kinds, in header order, and none of
lgu_corr.h's; lib() applies it; every _launch_ext / _lib.call_ext call in the package names one of them with the declared
number of arguments; call_ext refuses any other entry point."""
import ast
import ctypes
import glob
import os
import re

import pytest

from test_binding_cpu import PKG, ROOT, _ctype_kind, _kind


def _prototypes(header):
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", header)).read(), flags=re.S)
    out = []
    for ret, name, args in re.findall(r"LGU_API[ \t]+([^\n;(]*?)\s*\b(lgu_\w+)\s*\(([^)]*)\)\s*;", hdr):
        args = " ".join(args.split())
        kinds = [] if args in ("", "void") else [_kind(a) for a in args.split(",")]
        out.append((name, "pointer" if "*" in ret else ret.strip(), kinds))
    n_decl = sum(1 for line in hdr.splitlines() if line.startswith("LGU_API "))
    assert len(out) == n_decl, f"{header}: {n_decl} LGU_API declarations, {len(out)} parsed"
    return out


def _binding():
    import lgu_slam_b200
    return lgu_slam_b200._lib


def test_ext_table_matches_the_ext_header():
    protos = _prototypes("lgu_corr_ext.h")
    assert "lgu_offset_heads_backward" in [p[0] for p in protos]
    table = _binding().EXT_SIGNATURES
    assert [s[0] for s in table] == [p[0] for p in protos], "one entry per prototype, in header order"
    for (name, ret, kinds), (_, argtypes, *rt) in zip(protos, table):
        assert [_ctype_kind(t) for t in argtypes] == kinds, name
        assert _ctype_kind(rt[0] if rt else ctypes.c_int) == ret, name
    base = {p[0] for p in _prototypes("lgu_corr.h")}
    assert not base & {p[0] for p in protos}, "an entry point is declared in one header only"


def test_lib_binds_the_ext_entry_points():
    b = _binding()
    if not os.path.exists(b.LIB_PATH):
        b.build()
    L = b.lib()
    for name, argtypes, *rt in b.EXT_SIGNATURES:
        fn = getattr(L, name)
        assert tuple(fn.argtypes) == tuple(argtypes), name
        assert fn.restype is (rt[0] if rt else ctypes.c_int), name


def test_every_ext_call_site_names_a_declared_entry_point_with_its_argument_count():
    declared = {name: len(argtypes) for name, argtypes, *_ in _binding().EXT_SIGNATURES}
    seen = 0
    for path in sorted(glob.glob(os.path.join(PKG, "**", "*.py"), recursive=True)):
        tree = ast.parse(open(path).read(), path)
        skip = set()
        for fn in ast.walk(tree):                # the forwarding body of _launch_ext itself
            if isinstance(fn, ast.FunctionDef) and fn.name == "_launch_ext":
                skip.update(id(n) for n in ast.walk(fn))
        for node in ast.walk(tree):
            if not isinstance(node, ast.Call) or id(node) in skip:
                continue
            f = node.func
            if isinstance(f, ast.Name) and f.id == "_launch_ext":
                fixed, extra = 2, 1
            elif isinstance(f, ast.Attribute) and f.attr == "call_ext" and isinstance(f.value, ast.Name) \
                    and f.value.id == "_lib":
                fixed, extra = 1, 0
            else:
                continue
            where = f"{os.path.relpath(path, ROOT)}:{node.lineno}"
            first = node.args[0] if node.args else None
            assert not node.keywords and not any(isinstance(a, ast.Starred) for a in node.args) and \
                isinstance(first, ast.Constant) and isinstance(first.value, str), f"{where}: call not countable"
            assert first.value in declared, f"{where}: {first.value} is not in EXT_SIGNATURES"
            assert len(node.args) - fixed + extra == declared[first.value], f"{where}: wrong argument count"
            seen += 1
    assert seen >= 1, "the scan must see the operator layer's calls"


def test_call_ext_refuses_other_entry_points():
    with pytest.raises(KeyError, match="not an entry point of lgu_corr_ext.h"):
        _binding().call_ext("lgu_offset_heads", None, None, None, None, None, 0, 98, 48, 64, 1e-5, None)
