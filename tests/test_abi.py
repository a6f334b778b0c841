"""The C-ABI library loads and exports every symbol include/toast_b200.h declares, with the
argument lists the ctypes binding assumes.  No compute calls (runs without a GPU)."""

import ctypes as ct
import os
import re

import pytest

from toast_b200 import build as tb_build
from toast_b200 import lib as tbl

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "toast_b200.h")

_CT = {
    "int64_t": tbl.I64, "int32_t": tbl.I32, "uint8_t": tbl.U8, "double": tbl.F64,
    "int": tbl.INT, "size_t": tbl.SZ, "uint64_t": ct.c_uint64,
}


def _parse_header():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", " ", src, flags=re.S)
    src = re.sub(r"//.*", " ", src)
    src = re.sub(r"typedef struct \{.*?\} \w+;", " ", src, flags=re.S)
    src = re.sub(r"enum \{.*?\};", " ", src, flags=re.S)
    protos = {}
    for m in re.finditer(r"([\w\s\*]+?)\b(tb_\w+)\s*\(([^;{}]*?)\)\s*;", src, flags=re.S):
        ret, name, args = m.group(1).strip(), m.group(2), m.group(3).strip()
        argl = [] if args in ("void", "") else [a.strip() for a in args.split(",")]
        protos[name] = (ret, argl)
    return protos


def _ctype_of(decl):
    if "*" in decl:
        return tbl.P
    toks = [t for t in decl.replace("const", " ").split() if t]
    return _CT[toks[0]]


def test_library_builds():
    path = tb_build.build()
    assert os.path.exists(path)


def test_every_declared_symbol_is_exported_and_bound():
    protos = _parse_header()
    assert len(protos) >= 40
    lib = tbl.load()
    for name, (ret, args) in protos.items():
        assert hasattr(lib, name), f"{name} not exported"
        assert name in tbl.PROTOTYPES, f"{name} has no ctypes prototype"
        res, argtypes = tbl.PROTOTYPES[name]
        assert len(argtypes) == len(args), (name, len(argtypes), len(args))
        for i, (decl, at) in enumerate(zip(args, argtypes)):
            want = _ctype_of(decl)
            if want is tbl.P:
                assert at in (tbl.P, tbl.STR) or issubclass(at, ct._Pointer), (name, i, decl)
            else:
                assert at is want, (name, i, decl, at)
    # and nothing bound that the header does not declare
    assert set(tbl.PROTOTYPES) == set(protos)


def test_runtime_queries_work_without_gpu():
    lib = tbl.load()
    assert b"toast_b200" in lib.tb_version()
    assert lib.tb_launch_count() >= 0
    assert lib.tb_accel_enabled() in (0, 1)


def test_removed_lhs_options_are_unknown():
    """The LHS paths that only an option could reach are gone, and so are their switches."""
    lib = tbl.load()
    for name in (b"tma", b"compact", b"sorted", b"sorted2"):
        assert lib.tb_get_option(name) == -1, name
        assert lib.tb_set_option(name, 1) == tbl.TB_ERR_ARG, name
        assert "unknown option" in tbl.last_error()
    for name in (b"blocked", b"crossings", b"pair", b"pairw"):
        assert lib.tb_get_option(name) in (0, 1), name


def test_no_cpu_fallback():
    """Without a device every compute entry point must fail loudly, not compute on the CPU."""
    import numpy as np

    lib = tbl.load()
    if lib.tb_accel_enabled():
        pytest.skip("a CUDA device is present")
    a = np.zeros(4)
    f = np.zeros(4, dtype=np.uint8)
    rc = lib.tb_template_offset_apply_diag_precond(a.ctypes.data, a.ctypes.data, f.ctypes.data,
                                                   a.ctypes.data, 4, tbl.TB_MEM_HOST, None)
    assert rc == tbl.TB_ERR_NO_DEVICE
    assert "no usable CUDA device" in tbl.last_error()
    with pytest.raises(RuntimeError):
        tbl.check(rc)
