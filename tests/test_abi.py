"""CPU: the C-ABI library loads and exports every symbol include/fcdiff_b200.h
declares; the ctypes table covers exactly that set.  No compute calls."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "fcdiff_b200.h")


def declared_symbols():
    src = open(HEADER).read()
    return sorted(set(re.findall(r"FCD_API\s+[\w\s\*]+?\b(fcd_\w+)\s*\(", src)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__
    __graft_entry__.build()
    from fcdiff_b200 import _lib
    return _lib


def test_header_declares_entry_points():
    syms = declared_symbols()
    assert len(syms) >= 30
    for must in ("fcd_estep_qF", "fcd_estep_qR", "fcd_elm_obj_grad", "fcd_energy_terms",
                 "fcd_mstep_stats", "fcd_sample_B_tilde", "fcd_corr_fisherz"):
        assert must in syms
    # one entry point per step: missing entries (S0 / `missing`) and the coded E-step's solver state are
    # arguments, not separate `_masked` / `_solved` symbols
    assert not [s for s in syms if s.endswith(("_masked", "_solved"))]


def test_library_exports_every_declared_symbol(lib):
    cdll = ctypes.CDLL(lib.LIB_PATH)
    for name in declared_symbols():
        assert hasattr(cdll, name), "missing export %s" % name


def test_ctypes_table_matches_header(lib):
    assert sorted(lib.SIGNATURES) == declared_symbols()


def test_load_and_version(lib):
    l = lib.load()
    assert l.fcd_version() >= 100
    assert l.fcd_workspace_bytes() > 0
    assert l.fcd_launch_count() >= 0
    assert l.fcd_corr_workspace_bytes(2, 8, 100) >= 2 * 8 * 100 * 4


def test_header_cites_reference_lines():
    src = open(HEADER).read()
    assert len(re.findall(r"fcdiff/(fit|model|util)\.py:\d+", src)) >= 15


def test_theta_struct_layout(lib):
    assert ctypes.sizeof(lib.FcdTheta) == 12 * 8


def _prototypes():
    """name -> parameter count of every FCD_API prototype in the header."""
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    out = {}
    for m in re.finditer(r"FCD_API\s+[\w\s\*]+?\b(fcd_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S):
        args = m.group(2).strip()
        out[m.group(1)] = 0 if args in ("", "void") else len([a for a in args.split(",") if a.strip()])
    return out


def test_ctypes_argument_counts_match_the_prototypes(lib):
    protos = _prototypes()
    assert sorted(protos) == declared_symbols()
    for (name, (_, argtypes)) in lib.SIGNATURES.items():
        assert len(argtypes) == protos[name], "%s: ctypes table has %d arguments, the header %d" % (
            name, len(argtypes), protos[name])
