"""Pin the C restatement (oracle/liboracle.so) to the compiled reference (oracle/_ref/libref.so).

The reference ships no golden vectors (SURVEY.md section 4), so the pin is the reference itself,
called function by function on seeded random inputs -- or, where it is not built, its answers on the same
inputs as recorded in tests/golden (oracle_lib.reference).  CPU only.
"""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as ol


@pytest.fixture(scope="module")
def tab():
    return ol.ref_tables()


@pytest.fixture(scope="module")
def mat():
    return ol.default_mat()


@pytest.mark.parametrize("model", ["generic", "mammal", "none"])
def test_nasw_global_cigar(tab, mat, model):
    rng = np.random.default_rng(101)
    par = dict(ol.DEFAULT_NASW)
    par["sp"] = {"generic": (8, 15, 21, 30, 0, 0), "mammal": (8, 15, 21, 30, 4, 4), "none": (0,) * 6}[model]
    n_ins = 0
    for it in range(250):
        nt, aa = ol.random_dp_problem(rng, al_max=70 if it % 5 else 180)
        a = ol.ref_nasw(nt, aa, 1, mat, par)
        b = ol.ora_nasw(tab, nt, aa, 1, mat, par)
        assert a[0] == b[0] and a[3] == b[3], (it, len(nt), len(aa), a, b)
        n_ins += any((c & 0xf) == 1 for c in a[3])
    assert n_ins > 10  # the segment-restart rule for insertions is exercised


@pytest.mark.parametrize("flag", [4, 2])
def test_nasw_extension(tab, mat, flag):
    rng = np.random.default_rng(202 + flag)
    par = dict(ol.DEFAULT_NASW)
    for it in range(250):
        nt, aa = ol.random_dp_problem(rng, al_max=60, flank=200)
        if len(nt) < 3:
            continue
        if it % 3 == 0:  # truncate so that the protein end is not always reachable
            nt = nt[:max(3, len(nt) // 2)] if flag == 4 else nt[len(nt) // 2:]
            if len(nt) < 3:
                continue
        if it % 7 == 0:
            par["io"] = 19
        else:
            par["io"] = 29
        a = ol.ref_nasw(nt, aa, flag, mat, par)
        b = ol.ora_nasw(tab, nt, aa, flag, mat, par)
        assert a[:3] == b[:3], (it, len(nt), len(aa), a, b)


def test_nasw_xdrop_fires(tab, mat):
    """Long junk tail after the gene: the reference must stop by x-drop and so must the restatement."""
    rng = np.random.default_rng(5)
    par = dict(ol.DEFAULT_NASW, xdrop=30)
    fired = 0
    for it in range(40):
        nt, aa = ol.random_dp_problem(rng, al_max=30, intron_max=0, flank=0)
        nt = np.concatenate([nt, np.full(600, 4, np.uint8)])  # N tail: no intron signal, scores decay
        a = ol.ref_nasw(nt, aa, 4, mat, par)
        b = ol.ora_nasw(tab, nt, aa, 4, mat, par)
        assert a[:3] == b[:3]
        fired += a[1] < len(nt) - 300
    assert fired > 0


def test_nasw_spsc_bytes(tab, mat):
    rng = np.random.default_rng(77)
    par = dict(ol.DEFAULT_NASW, io=39)
    for it in range(60):
        nt, aa = ol.random_dp_problem(rng, al_max=50)
        if len(nt) < 3:
            continue
        ss = np.full(len(nt), 0xff, np.uint8)
        k = rng.random(len(nt)) < 0.05
        ss[k] = ((rng.integers(-10, 20, size=int(k.sum())) + 64) << 1 | rng.integers(0, 2, size=int(k.sum()))).astype(np.uint8)
        for flag in (1, 2, 4):
            a = ol.ref_nasw(nt, aa, flag, mat, par, ss)
            b = ol.ora_nasw(tab, nt, aa, flag, mat, par, ss)
            assert a[0] == b[0] and (a[3] == b[3] if flag == 1 else a[:3] == b[:3]), (it, flag, a, b)


def test_sort128x_matches_reference_permutation():
    rng = np.random.default_rng(9)
    o = ol.ora()
    for n in (1, 2, 63, 64, 65, 200, 1000, 5000, 70000):
        for hi in (3, 50, 1 << 20):
            z = np.zeros((n, 2), np.uint64)
            z[:, 0] = rng.integers(0, hi, size=n)
            z[:, 1] = np.arange(n)
            b = z.copy()
            o.ora_sort128x(b.ctypes.data_as(C.c_void_p), C.c_void_p(b.ctypes.data + 16 * n))
            assert ol.digest(b.tobytes()) == ol.ref_sort128x(z), (n, hi)
            assert (np.diff(b[:, 0].astype(np.int64)) >= 0).all()


def test_hash_and_sketch(tab):
    rng = np.random.default_rng(3)
    o = ol.ora()
    for it in range(40):
        L = int(rng.integers(1, 600))
        alpha = b"ARNDCQEGHILKMFPSTWYV" + (b"X*" if it % 3 == 0 else b"")
        seq = bytes(alpha[i] for i in rng.integers(0, len(alpha), size=L))
        for k, m in ((6, 1), (5, 0)):
            out = np.zeros(L + 1, np.uint64)
            n = o.ora_sketch_prot(C.byref(tab), seq, L, k, m, out.ctypes.data_as(C.c_void_p))
            assert (n, ol.digest(out[:n].tobytes())) == ol.ref_sketch_prot(seq, k, m)
    for it in range(30):
        L = int(rng.integers(50, 6000))
        nt = rng.integers(0, 4, size=L).astype(np.uint8)
        if it % 2:  # thin out stops so that long ORFs exist
            for s in range(0, L - 2, 3):
                if nt[s] == 3 and ((nt[s + 1] == 0 and nt[s + 2] in (0, 2)) or (nt[s + 1] == 2 and nt[s + 2] == 0)):
                    nt[s] = 1
        if it % 4 == 0:
            nt[rng.random(L) < 0.003] = 4
        for (k, m, bbit, boff) in ((6, 1, 8, 1234), (5, 0, 0, 0)):
            out = np.zeros(L + 1, np.uint64)
            n = o.ora_sketch_nt4(C.byref(tab), nt.ctypes.data_as(C.c_void_p), C.c_int64(L), 30, k, m, bbit, C.c_int64(boff),
                                 out.ctypes.data_as(C.c_void_p))
            want = ol.ref_sketch_nt4(nt, k, m, bbit, boff)
            assert (n, ol.digest(out[:n].tobytes())) == want, (it, k, n, want[0])


@pytest.mark.parametrize("mode", ["pre", "main", "refine"])
def test_chain(mode):
    rng = np.random.default_rng({"pre": 11, "main": 12, "refine": 13}[mode])
    n_nonempty = 0
    for it in range(120):
        n = int(rng.integers(1, 60 if it % 4 else 900))
        a = ol.random_chain_problem(rng, n, mode)
        over = {}
        if it % 10 == 0:
            over = dict(is_spliced=0, bw=500, max_dist_x=500)
        if it % 13 == 0:
            over["max_skip"] = 2
        par = ol.chain_par(mode, **over)
        ua, ba = ol.ref_chain(par, a)
        ub, bb = ol.ora_chain(par, a)
        assert len(ua) == len(ub) and (ua == ub).all() and (ba == bb).all(), (mode, it, n)
        n_nonempty += len(ua) > 0
    assert n_nonempty > 30


def _random_scoring(rng, go_min=1):
    """Scoring parameters over the range the CLI reaches (-O -E -J -F -B, splice models, x-drop, ie_coef)."""
    par = dict(ol.DEFAULT_NASW)
    par.update(go=int(rng.integers(go_min, 31)), ge=int(rng.integers(0, 6)), io=int(rng.integers(3, 61)), fs=int(rng.integers(1, 61)),
               end_bonus=int(rng.integers(0, 21)), xdrop=int(rng.choice([5, 30, 100, 400])), ie_coef=float(rng.choice([0.0, 0.25, 0.5, 1.0, 2.5])))
    if rng.random() < 0.5:
        par["sp"] = tuple(int(x) for x in rng.integers(0, 40, size=4)) + (int(rng.integers(0, 8)), int(rng.integers(0, 8)))
    return par


def test_nasw_random_scoring_parameters(tab):
    """The restatement equals the reference for every gap-open penalty >= 1 together with random other penalties, stop-codon
    scores (-C, options.c:87-88) and problem shapes (tools/fuzz_emu.py runs the same comparison open-ended)."""
    rng = np.random.default_rng(909)
    for it in range(150):
        par = _random_scoring(rng)
        m = ol.default_mat()
        if it % 3 == 0:
            ol.ref_set_stop_sc(m, int(rng.integers(1, 60)))
        nt, aa = ol.random_dp_problem(rng, al_max=int(rng.choice([12, 64, 140, 300])), flank=int(rng.choice([0, 3, 60])),
                                      intron_max=int(rng.choice([0, 60, 400])), p_sub=float(rng.choice([0.05, 0.2, 0.5])))
        if len(nt) < 3:
            continue
        for flag in (1, 4, 2):
            b = ol.ora_nasw(tab, nt, aa, flag, m, par)
            if flag != 1 and b[2] == len(aa) + 1:
                continue  # the reference stops at an assertion here (nasw-sse.c:441)
            a = ol.ref_nasw(nt, aa, flag, m, par)
            assert (a[0] == b[0] and a[3] == b[3]) if flag == 1 else (a[:3] == b[:3]), (it, flag, len(nt), len(aa), par, a[:3], b[:3])


def test_nasw_gap_open_zero_is_layout_dependent_in_the_reference(tab, mat):
    """go == 0 is outside the restatement (oracle/nasw.c header) and refused by the product: the reference's lazy-F loop
    (nasw-sse.c:408-422) then stops after the first stripe, so its scores fall BELOW the recurrence's on some problems --
    never above, and never for go >= 1.  Pins the reason for the precondition."""
    rng = np.random.default_rng(4)
    below = 0
    for it in range(200):
        par = _random_scoring(rng)
        par["go"] = 0
        nt, aa = ol.random_dp_problem(rng, al_max=80, flank=30)
        if len(nt) < 3:
            continue
        a, b = ol.ref_nasw(nt, aa, 1, mat, par), ol.ora_nasw(tab, nt, aa, 1, mat, par)
        assert a[0] <= b[0], (it, a[0], b[0])
        below += a[0] < b[0]
    assert below > 0


def test_committed_goldens_are_what_the_reference_prints(tmp_path):
    """tests/golden/*.paf are the reference's own output (tests/golden/make_golden.py): compare them with what the compiled reference
    prints on the same inputs (run here, or as recorded), so that a stale or hand-edited golden cannot pass for the reference."""
    import hashlib
    import os

    from miniprot_b200 import synth

    gold = ol.GOLDEN

    def same(args, g, p, name):
        want = ol.ref_cli(args, g, p)
        return hashlib.md5(open(os.path.join(gold, name), "rb").read()).hexdigest() == want["md5"]

    g, p = ol.DPP3_GEN, ol.DPP3_PEP
    assert ol.ref_cli([], g, p)["md5"] == "74fd00200bda6c03380bb3062fb5178b"  # SURVEY.md App. D
    assert same([], g, p, "DPP3_default.paf")
    assert same(["-j2"], g, p, "DPP3_j2.paf")
    assert same(["--gff"], g, p, "DPP3_gff.txt")
    for cfg in ("tiny", "tiny5"):
        gg, pp = synth.generate(synth.CONFIGS[cfg], str(tmp_path))
        assert same([], gg, pp, cfg + ".paf")
    gg, pp = synth.generate(synth.CONFIGS["tiny5"], str(tmp_path))
    assert same(["--gtf"], gg, pp, "tiny5_gtf.txt")
