"""The C-ABI library builds, loads and exports every symbol include/lcao_b200.h declares (no compute)."""
import ctypes
import os
import re

import pytest
import torch

from lcaonet_b200 import _lib
from lcaonet_b200.csrc.build import build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "lcao_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(lcao_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(build())
    names = _declared()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), n
    lib.lcao_version.restype = ctypes.c_int
    assert lib.lcao_version() >= 100


def test_python_signatures_cover_the_header():
    declared = set(_declared()) - {"lcao_version", "lcao_last_error", "lcao_launch_count", "lcao_linear_bwd_scratch",
                                   "lcao_pair_contract_bwd_scratch"}
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    text = open(os.path.join(ROOT, "include", "lcao_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    for name, argtypes in _lib.SIGNATURES.items():
        m = re.search(r"\b" + name + r"\s*\((.*?)\)\s*;", text, flags=re.S)
        assert m, name
        assert len([a for a in m.group(1).split(",") if a.strip()]) == len(argtypes), name


def test_basis_spec_layout_matches_header():
    # 4 int32 + 2 double + 3*18 int32 + 18 double + 18*8 double
    assert ctypes.sizeof(_lib.BasisSpec) == 16 + 16 + 3 * 18 * 4 + 18 * 8 + 18 * 8 * 8


def test_argument_errors_are_reported_without_a_gpu():
    lib = _lib.load()
    rc = lib.lcao_twobody_fwd(None, 3, None, 10, 128, 3, 0, None, None)
    assert rc == -1 and b"null buffer" in lib.lcao_last_error()
    rc = lib.lcao_threebody_fwd(1, 3, 1, 1, 1, 8, 1, 1, 1, 1, 1, 4, 4, 130, 3, 1, None)
    assert rc == -1 and b"C % 4" in lib.lcao_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="without the check, a GPU would run the kernels on these addresses")
def test_threebody_rejects_unaligned_rows():
    # pointer values only: every kernel reads B, gate, d_tbw and dP and writes tbw, dB and q with 16-byte accesses or
    # bulk copies.  Each case misaligns one pointer; C = 128 and C = 256 reach both kernel families' entry points.
    lib = _lib.load()
    a, odd = 16, 4
    for C in (128, 256):
        for B, gate, tbw in ((odd, a, a), (a, odd, a), (a, a, odd)):
            rc = lib.lcao_threebody_fwd(B, 3, a, a, gate, C, a, a, a, a, a, 4, 4, C, 3, tbw, None)
            assert rc == -1 and b"aligned" in lib.lcao_last_error(), (C, B, gate, tbw)
        bwd = dict(B=a, gate=a, d_tbw=a, dP=a, dB=a, q=a)
        for name in bwd:
            p = dict(bwd, **{name: odd})
            rc = lib.lcao_threebody_bwd(p["B"], 3, a, a, p["gate"], C, a, a, a, a, a, 4, 4, C, 3, p["d_tbw"], p["dP"], p["dB"],
                                        p["q"], None, None, None)
            assert rc == -1 and b"aligned" in lib.lcao_last_error(), (C, name)


@pytest.mark.skipif(torch.cuda.is_available(), reason="without the check, a GPU would run the kernels on these addresses")
def test_edge_basis_rejects_unaligned_rows_and_unknown_kinds():
    # pointer values only, as above: the contraction kernels read tab / cst1 / dB and write B / psum / d_tab / d_cst1 and
    # the keyed-reduction partials with 16-byte accesses.  Each case misaligns one pointer; C = 128 and C = 256 reach both
    # d_rb kernels of lcao_pair_contract_bwd.
    lib = _lib.load()
    a, odd = 16, 4
    E, O, NL = 64, 8, 2
    for C in (128, 256):
        fwd = dict(tab=a, B=a, psum=a)
        for name in fwd:
            p = dict(fwd, **{name: odd})
            rc = lib.lcao_pair_contract_fwd(p["tab"], a, a, a, a, E, O, C, NL, 1, p["B"], a, p["psum"], None)
            assert rc == -1 and b"aligned" in lib.lcao_last_error(), (C, name)
        bwd = dict(tab=a, dB=a, d_tab=a, scratch=a)
        for name in bwd:
            p = dict(bwd, **{name: odd})
            rc = lib.lcao_pair_contract_bwd(p["tab"], a, a, a, a, a, a, p["dB"], E, 9, O, C, NL, 1, p["d_tab"], a,
                                            p["scratch"], None)
            assert rc == -1 and b"aligned" in lib.lcao_last_error(), (C, name)
        # tab is read only for d_rb: d_tab alone accepts it misaligned (the call then fails only at the launch)
        rc = lib.lcao_pair_contract_bwd(odd, a, a, a, a, a, a, a, E, 9, O, C, NL, 1, a, None, a, None)
        assert b"aligned" not in lib.lcao_last_error()
        # d_rb without tab is rejected before d_tab is written
        rc = lib.lcao_pair_contract_bwd(None, a, a, a, a, a, a, a, E, 9, O, C, NL, 1, a, a, a, None)
        assert rc == -1 and b"d_rb needs tab" in lib.lcao_last_error(), C
        rc = lib.lcao_coeff_contract_fwd(odd, a, a, a, E, O, C, NL, 1, a, None)
        assert rc == -1 and b"aligned" in lib.lcao_last_error(), C
        rc = lib.lcao_coeff_contract_fwd(a, a, a, a, E, O, C, NL, 1, odd, None)
        assert rc == -1 and b"aligned" in lib.lcao_last_error(), C
        cbwd = dict(cst1=a, dB=a, d_cst1=a)
        for name in cbwd:
            p = dict(cbwd, **{name: odd})
            rc = lib.lcao_coeff_contract_bwd(p["cst1"], a, a, a, p["dB"], E, O, C, NL, 1, p["d_cst1"], a, None)
            assert rc == -1 and b"aligned" in lib.lcao_last_error(), (C, name)

    sp = _lib.BasisSpec()
    sp.n_unique, sp.n_rep, sp.rc, sp.a0 = 1, 1, 5.0, 0.529
    sp.n[0], sp.l[0], sp.deg[0], sp.norm[0], sp.poly[0][0] = 1, 0, 0, -1.0, -1.0
    for cut, rbf in ((3, 0), (-1, 0), (0, 2), (2, -1)):
        sp.cutoff_kind, sp.rbf_kind = cut, rbf
        rc = lib.lcao_geom_basis_fwd(a, a, a, None, a, a, E, ctypes.byref(sp), a, a, a, None, None)
        assert rc == -1 and b"unknown" in lib.lcao_last_error(), (cut, rbf)


@pytest.mark.skipif(torch.cuda.is_available(), reason="without the check, a GPU would run the kernels on these addresses")
def test_message_entry_points_reject_bad_flags_activations_and_alignment():
    # pointer values only: every case must be refused before the first launch
    lib = _lib.load()
    a, odd = 16, 4
    R, C = 4, 128
    for mode, y in ((2 | 4, a), (2, None), (4, None), (4 | (5 << 4), None), (8, a), (1 << 8, a), (1 << 12, a), (-1, a)):
        rc = lib.lcao_segment_sum(a, C, y, C, a, a, R, C, mode, a, C, None)
        assert rc == -1 and b"flag word" in lib.lcao_last_error(), (mode, y)
    # an edge-less batch passes neither x nor y: nothing is read, so bit 1 or 2 is accepted (it then fails at the launch)
    rc = lib.lcao_segment_sum(None, C, None, C, a, a, R, C, 2 | (1 << 4), a, C, None)
    assert b"flag word" not in lib.lcao_last_error()
    E = 64
    for bias, pre in ((odd, a), (a, odd), (odd, None)):
        rc = lib.lcao_edge_pair_fwd(a, C, a, C, bias, a, a, E, C, 1, a, pre, None)
        assert rc == -1 and b"aligned" in lib.lcao_last_error(), (bias, pre)
    for act in (-1, 10, 1 << 20):
        rc = lib.lcao_edge_pair_fwd(a, C, a, C, a, a, a, E, C, act, a, a, None)
        assert rc == -1 and b"activation" in lib.lcao_last_error(), act
        for width in (C, 127):   # the vector and the any-alignment kernel
            rc = lib.lcao_act_bwd(a, width, a, width, a, width, R, width, act, None)
            assert rc == -1 and b"activation" in lib.lcao_last_error(), (act, width)
