"""CPU: the C-ABI library loads, exports every symbol include/mobocmf_b200.h declares, and the ctypes signatures
agree with the header's parameter counts (no compute calls: there is no GPU here)."""
import os
import re

from mobocmf_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "mobocmf_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    out = {}
    for m in re.finditer(r"\b(?:int|size_t|void\s*\*|void|long long)\s*(mobo_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S):
        args = m.group(2).strip()
        out[m.group(1)] = 0 if args in ("", "void") else len(args.split(","))
    return out


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    decl = header_functions()
    assert len(decl) >= 12
    for name in decl:
        assert hasattr(lib, name), name
    assert lib.mobo_abi_version() == 103


def test_ctypes_signatures_match_header():
    decl = header_functions()
    for name, (res, args) in _lib._SIGNATURES.items():
        assert name in decl, name
        assert len(args) == decl[name], (name, len(args), decl[name])
    assert set(decl) == set(_lib._SIGNATURES)


def test_size_queries():
    lib = _lib.load()
    assert lib.mobo_padded_m(16) == 32 and lib.mobo_padded_m(256) == 256 and lib.mobo_padded_m(75) == 96
    assert lib.mobo_ops_doubles(256) == 11 * 256 * 256 + 6 * 256 + 16 + 128
    assert lib.mobo_rows_save_doubles(256, 65536) == 65536 * 256
    assert lib.mobo_rows_save_doubles(16, 10) == 32 * 32
