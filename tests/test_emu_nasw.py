"""CPU lock-step emulation of the nasw CUDA kernels (same per-lane header the kernels compile) vs the oracle."""
import ctypes as C

import numpy as np
import pytest

import build_hostcheck
import oracle_lib as ol


@pytest.fixture(scope="module")
def hc():
    lib = C.CDLL(build_hostcheck.build())
    lib.emu_nasw.restype = C.c_int
    lib.emu_nasw.argtypes = [C.c_void_p] * 5 + [C.c_int] * 6 + [C.c_float, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_char_p, C.c_int] + \
        [C.c_void_p] * 4 + [C.c_int]
    return lib


def emu(hc, nt, aa, flag, Ccols, mat, par):
    tab = ol.ref_tables()
    sp = (C.c_int32 * 6)(*par["sp"])
    sc, ntl, aal = C.c_int(), C.c_int(), C.c_int()
    cig = (C.c_uint32 * (len(nt) + len(aa) + 16))()
    n = hc.emu_nasw(tab.nt4, tab.aa20, tab.codon, mat.ctypes.data, C.addressof(sp), par["go"], par["ge"],
                    par["io"], par["fs"], par["xdrop"], par["end_bonus"], par["ie_coef"], flag, Ccols,
                    nt.ctypes.data, len(nt), aa, len(aa), C.addressof(sc), C.addressof(ntl), C.addressof(aal), C.addressof(cig), len(cig))
    return sc.value, ntl.value, aal.value, [cig[i] for i in range(n)]


@pytest.mark.parametrize("Ccols", [-1, 0, 1, 2, 4, 8])  # 0 = block-wide wavefront kernels (one thread per column, 3 rows per step); -1 = pair-lane kernels (int16x2)
def test_emu_matches_oracle(hc, Ccols):
    rng = np.random.default_rng(1000 + Ccols)
    tab, mat = ol.ref_tables(), ol.default_mat()
    for it in range(120):
        par = dict(ol.DEFAULT_NASW)
        if it % 5 == 0:
            par["sp"] = (8, 15, 21, 30, 4, 4)
        al_max = (250, 250, 30, 70, 140, 300)[[-1, 0, 1, 2, 4, 8].index(Ccols)]
        if it % 6 == 0 and Ccols >= 0:
            al_max = 32 * Ccols * 2 + 20 if Ccols else (700 if it % 12 else 560)  # force several column passes (256 columns each when Ccols == 0)
        nt, aa = ol.random_dp_problem(rng, al_max=al_max, flank=60)
        if len(nt) < 3:
            continue
        for flag in (1, 4, 2):
            if flag != 1 and it % 7 == 0:
                par["io"] = 19
            a = ol.ora_nasw(tab, nt, aa, flag, mat, par)
            b = emu(hc, nt, aa, flag, Ccols, mat, par)
            if flag == 1:
                assert a[0] == b[0] and a[3] == b[3], (it, flag, len(nt), len(aa), a, b)
            else:
                assert a[:3] == b[:3], (it, flag, len(nt), len(aa), a[:3], b[:3])


def test_emu_extension_wider_than_4095_columns(hc):
    """The row maximum carries its column in 15 bits once the extension has more than 4095 columns (nasw_core.cuh code_bits)."""
    rng = np.random.default_rng(77)
    tab, mat = ol.ref_tables(), ol.default_mat()
    par = dict(ol.DEFAULT_NASW)
    nt, aa = ol.random_dp_problem(rng, al_max=4400, flank=30, intron_max=200, p_sub=0.25)
    while len(aa) < 4200:
        nt, aa = ol.random_dp_problem(rng, al_max=4400, flank=30, intron_max=200, p_sub=0.25)
    for flag, Ccols in ((4, 0), (2, 8)):
        assert ol.ora_nasw(tab, nt, aa, flag, mat, par)[:3] == emu(hc, nt, aa, flag, Ccols, mat, par)[:3]


def test_emu_xdrop_and_tiny(hc):
    rng = np.random.default_rng(4)
    tab, mat = ol.ref_tables(), ol.default_mat()
    par = dict(ol.DEFAULT_NASW, xdrop=30)
    for it in range(30):
        nt, aa = ol.random_dp_problem(rng, al_max=30, intron_max=0, flank=0)
        nt = np.concatenate([nt, np.full(500, 4, np.uint8)])
        assert ol.ora_nasw(tab, nt, aa, 4, mat, par)[:3] == emu(hc, nt, aa, 4, 1, mat, par)[:3]
        assert ol.ora_nasw(tab, nt, aa, 4, mat, par)[:3] == emu(hc, nt, aa, 4, 0, mat, par)[:3]
    for nl in (0, 1, 2, 3, 4, 5):  # degenerate global problems (no DP rows for nl < 3)
        for al in (1, 2, 9):
            nt = rng.integers(0, 4, size=nl).astype(np.uint8)
            aa = bytes(b"ARNDCQEGH"[:al])
            for cc in (1, 0):
                a, b = ol.ora_nasw(tab, nt, aa, 1, mat, dict(ol.DEFAULT_NASW)), emu(hc, nt, aa, 1, cc, mat, dict(ol.DEFAULT_NASW))
                assert a[0] == b[0] and a[3] == b[3], (nl, al, cc, a, b)


def test_pen_table_equals_fp_formula(hc):
    hc.emu_pen_check.restype = C.c_int
    hc.emu_pen_check.argtypes = [C.c_float, C.c_int]
    for coef in (0.5, 0.25, 1.0, 3.0):  # PEN_STEPS covers ie_coef up to ~5
        assert hc.emu_pen_check(coef, 3_000_000) == 0


def test_emu_score_when_end_column_is_first_of_a_pass(hc):
    """Global score is read at (nl-1, al-1).  When al-1 is the FIRST column of a block or pass (al = 1, 257, 513) its last row
    comes earliest of all columns -- it must not fall into the check-free steady loop (regression: AS:i of one C5 hit)."""
    rng = np.random.default_rng(4242)
    tab, mat = ol.ref_tables(), ol.default_mat()
    par = dict(ol.DEFAULT_NASW)
    for al, nls in ((1, (104, 107, 110, 113, 116)), (257, (803, 806, 809, 812, 815)), (513, (806, 809, 812, 1211))):
        for nl in nls:
            nt0, aa = ol.random_dp_problem(rng, al_max=al, flank=10, intron_max=100)
            aa = (aa + bytes(b"ARNDCQEGHILKMFPSTWYV"[i] for i in rng.integers(0, 20, size=al)))[:al]
            nt = np.concatenate([nt0, rng.integers(0, 4, size=nl).astype(np.uint8)])[:nl]
            a = ol.ora_nasw(tab, nt, aa, 1, mat, par)
            b = emu(hc, nt, aa, 1, 0, mat, par)
            assert a[0] == b[0] and a[3] == b[3], (al, nl, a[0], b[0])


def random_spsc(rng, nt, max_sc=14, p_set=0.3):
    """--spsc bytes for a slice (ntseq.c:130-156): 0xff = unset, else (score + 64) << 1 | is_acceptor."""
    n = len(nt)
    ss = np.full(n, 0xff, dtype=np.uint8)
    k = rng.random(n) < p_set
    sc = rng.integers(-max_sc, max_sc + 1, n)
    ty = rng.integers(0, 2, n)
    ss[k] = ((sc[k] + 64) << 1 | ty[k]).astype(np.uint8)
    return ss


def emu_ss(hc, nt, aa, flag, Ccols, mat, par, ss):
    tab = ol.ref_tables()
    hc.emu_nasw_ss.restype = C.c_int
    hc.emu_nasw_ss.argtypes = [C.c_void_p] * 5 + [C.c_int] * 6 + [C.c_float, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_char_p, C.c_int] + \
        [C.c_void_p] * 4 + [C.c_int, C.c_void_p, C.c_int]
    sp = (C.c_int32 * 6)(*par["sp"])
    sc, ntl, aal = C.c_int(), C.c_int(), C.c_int()
    cig = (C.c_uint32 * (len(nt) + len(aa) + 16))()
    n = hc.emu_nasw_ss(tab.nt4, tab.aa20, tab.codon, mat.ctypes.data, C.addressof(sp), par["go"], par["ge"],
                       par["io"], par["fs"], par["xdrop"], par["end_bonus"], par["ie_coef"], flag, Ccols,
                       nt.ctypes.data, len(nt), aa, len(aa), C.addressof(sc), C.addressof(ntl), C.addressof(aal), C.addressof(cig), len(cig),
                       ss.ctypes.data, par["sp_null_bonus"])
    return sc.value, ntl.value, aal.value, [cig[i] for i in range(n)]


@pytest.mark.parametrize("Ccols", [0, 1, 8])
def test_emu_with_splice_scores_matches_reference(hc, Ccols):
    """--spsc (nasw-sse.c:138-152,189-203): donor / acceptor entries shifted by per-base scores, negative ones included.  The same
    per-row preparation the prep kernels compile, against the reference's own ns_global_gs16b and the oracle."""
    rng = np.random.default_rng(4242 + Ccols)
    tab, mat = ol.ref_tables(), ol.default_mat()
    for it in range(80):
        par = dict(ol.DEFAULT_NASW)
        par["io"] = 39 if it % 4 else 29          # mp_set_spsc adds 10 unless --spsc-keep-io (index.c:242)
        par["sp_null_bonus"] = -7 if it % 3 else -2
        nt, aa = ol.random_dp_problem(rng, al_max=(120, 30, 200)[[0, 1, 8].index(Ccols)], flank=60)
        if len(nt) < 3:
            continue
        ss = random_spsc(rng, nt, max_sc=(par["io"] + 1) // 2 - 1 if it % 5 else 40, p_set=0.3 if it % 2 else 0.9)
        for flag in (1, 4, 2):
            a = ol.ref_nasw(nt, aa, flag, mat, par, ss)
            o = ol.ora_nasw(tab, nt, aa, flag, mat, par, ss)
            b = emu_ss(hc, nt, aa, flag, Ccols, mat, par, ss)
            if flag == 1:
                assert a[0] == b[0] == o[0] and a[3] == b[3] == o[3], (it, flag, len(nt), len(aa), a, b)
            else:
                assert a[:3] == b[:3] == o[:3], (it, flag, len(nt), len(aa), a[:3], b[:3])


def test_emu_random_scoring_parameters():
    """Random problems x random scoring parameters (-O >= 1, -E, -J, -F, -B, -C, splice models, x-drop, ie_coef, --spsc bytes)
    through every kernel family -- the pair-lane family where the dispatcher's value-domain check admits the problem -- against
    the reference's ns_global_gs16b and the oracle.  A fixed-seed slice of tools/fuzz_emu.py (which runs open-ended)."""
    import os
    import sys

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import fuzz_emu

    n_cmp, n_pair, n_bad = fuzz_emu.fuzz(20260924, 80)
    assert n_bad == 0 and n_cmp > 400 and n_pair > 50


def test_emu_random_scoring_parameters_long_profile(monkeypatch):
    """The same comparison on the fuzzer's "long" profile: problems of several column passes (up to 1500 columns), thousands of rows,
    long introns, slices cut anywhere, runs of N."""
    import os
    import sys

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import fuzz_emu

    monkeypatch.setattr(fuzz_emu, "LONG", True)
    n_cmp, _, n_bad = fuzz_emu.fuzz(424242, 8)
    assert n_bad == 0 and n_cmp >= 30
