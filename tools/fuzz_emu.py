"""Differential fuzzing of the nasw kernels' per-thread code on the CPU (no GPU needed): random problems AND random scoring
parameters (-O/-E/-J/-F/-B/-C, splice models, x-drop, ie_coef) through the lock-step emulation of every kernel family
(tests/hostcheck/emu_nasw.cpp: the same nasw_core.cuh / nasw_pair.cuh the kernels compile) against the reference's own
ns_global_gs16b (oracle/_ref/libref.so) and the C oracle.  The pair-lane family is only asked about problems the dispatcher would
send it (emu_pair_eligible = nasw_host.cu use_pair).  Test infrastructure, not part of the product.

usage: python tools/fuzz_emu.py [seed] [n_iterations]"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import build_hostcheck  # noqa: E402
import oracle_lib as ol  # noqa: E402
from test_emu_nasw import emu, emu_ss, random_spsc  # noqa: E402


LONG = os.environ.get("MPB_FUZZ_PROFILE") == "long"


def random_par(rng):
    par = dict(ol.DEFAULT_NASW)
    if rng.random() < 0.7:
        par["go"] = int(rng.integers(1, 31))  # go == 0: outside the contract (backend.cu bad_scoring)
        par["ge"] = int(rng.integers(0, 6))
        par["io"] = int(rng.integers(3, 61))
        par["fs"] = int(rng.integers(1, 61))
        par["end_bonus"] = int(rng.integers(0, 21))
        par["xdrop"] = int(rng.choice([5, 30, 100, 400]))
        par["ie_coef"] = float(rng.choice([0.0, 0.25, 0.5, 1.0, 2.5]))
    if rng.random() < 0.5:
        par["sp"] = tuple(int(x) for x in rng.integers(0, 40, size=4)) + (int(rng.integers(0, 8)), int(rng.integers(0, 8)))
    return par


def fuzz(seed, n_it):
    hc = C.CDLL(build_hostcheck.build())
    hc.emu_nasw.restype = C.c_int
    hc.emu_nasw.argtypes = [C.c_void_p] * 5 + [C.c_int] * 6 + [C.c_float, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_char_p, C.c_int] + [C.c_void_p] * 4 + [C.c_int]
    hc.emu_pair_eligible.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int] * 7
    rng = np.random.default_rng(seed)
    tab = ol.ref_tables()
    n_cmp = n_pair = n_bad = 0
    for it in range(n_it):
        if it and it % (200 if LONG else 2000) == 0:
            print(f"progress seed {seed}: {it} problems, {n_cmp} comparisons ({n_pair} on the pair-lane family), {n_bad} mismatches", flush=True)
        par = random_par(rng)
        mat = ol.default_mat()
        if rng.random() < 0.3:  # -C: stop-codon score scale (options.c:87-88)
            ol.ref_set_stop_sc(mat, int(rng.integers(1, 60)))
        shape = rng.random()
        if LONG:  # MPB_FUZZ_PROFILE=long: several column passes, thousands of rows, long introns, slices cut anywhere
            al_max = 300 if shape < 0.4 else 700 if shape < 0.8 else 1500
            nt, aa = ol.random_dp_problem(rng, al_max=al_max, flank=int(rng.choice([0, 60, 2000])), intron_max=int(rng.choice([400, 5000])),
                                          p_sub=float(rng.choice([0.05, 0.2, 0.5])), p_fs=float(rng.choice([0.0, 0.02, 0.1])), p_n=float(rng.choice([0.0, 0.002, 0.05])))
            if rng.random() < 0.3 and len(nt) > 8:
                a, b = sorted(int(x) for x in rng.integers(0, len(nt), size=2))
                nt = nt[a:b] if b - a >= 3 else nt
        else:
            al_max = 12 if shape < 0.2 else 64 if shape < 0.6 else 140 if shape < 0.85 else 300 if shape < 0.97 else 600
            nt, aa = ol.random_dp_problem(rng, al_max=al_max, flank=int(rng.choice([0, 3, 60])), intron_max=int(rng.choice([0, 60, 400])),
                                          p_sub=float(rng.choice([0.05, 0.2, 0.5])), p_fs=float(rng.choice([0.0, 0.02, 0.1])))
            if rng.random() < 0.1:
                nt = nt[:int(rng.integers(0, 8))]
            elif rng.random() < 0.1 and len(nt) > 8:
                a, b = sorted(int(x) for x in rng.integers(0, len(nt), size=2))
                nt = nt[a:b] if b - a >= 3 else nt
        use_ss = rng.random() < 0.15
        ss = random_spsc(rng, nt, max_sc=(par["io"] + 1) // 2 - 1 if rng.random() < 0.7 else 40) if use_ss and len(nt) else None
        sp = (C.c_int32 * 6)(*par["sp"])
        for flag in (1, 4, 2):
            o = ol.ora_nasw(tab, nt, aa, flag, mat, par, ss)
            # an extension whose best row has its maximum nowhere in the real columns: the reference stops at an assertion
            # (nasw-sse.c:441), the oracle reports aa_len = al + 1 -- the product has to agree with the oracle there
            want = o if flag != 1 and (o[2] == len(aa) + 1 or len(nt) < 3) else ol.ref_nasw(nt, aa, flag, mat, par, ss)
            fams = [0, int(rng.choice([1, 2, 4, 8]))]
            if ss is None and hc.emu_pair_eligible(mat.ctypes.data, C.addressof(sp), par["go"], par["ge"], par["io"], par["fs"], par["end_bonus"], len(nt), len(aa)):
                fams.append(-1)
                n_pair += 1
            for fam in fams:
                got = emu_ss(hc, nt, aa, flag, fam, mat, par, ss) if ss is not None else emu(hc, nt, aa, flag, fam, mat, par)
                n_cmp += 1
                if len(nt) < 3 and flag != 1:
                    continue  # nothing to extend into (the reference asserts, nasw-sse.c:443)
                ok = (want[0] == got[0] == o[0] and want[3] == got[3] == o[3]) if flag == 1 else (want[:3] == got[:3] == o[:3])
                if not ok:
                    n_bad += 1
                    print(f"MISMATCH seed={seed} it={it} flag={flag} family={fam} nl={len(nt)} al={len(aa)} par={par} ss={ss is not None}\n  ref={want[:3]} ora={o[:3]} emu={got[:3]}", flush=True)
    print(f"seed {seed}: {n_cmp} comparisons ({n_pair} on the pair-lane family), {n_bad} mismatches", flush=True)
    return n_cmp, n_pair, n_bad


if __name__ == "__main__":
    sys.exit(1 if fuzz(int(sys.argv[1]) if len(sys.argv) > 1 else 1, int(sys.argv[2]) if len(sys.argv) > 2 else 300)[2] else 0)
