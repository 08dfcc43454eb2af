"""ctypes bindings for the two CHECKERS (test infrastructure only):

* ``oracle/_ref/libref.so``  - the unmodified reference, every symbol renamed ``ref_*``
* ``oracle/liboracle.so``    - the plain-C restatement of the hot path

plus seeded random problem generators shared by the CPU and GPU parity tests.

Every answer of the reference goes through ``reference()``: where oracle/_ref is built the reference is called, elsewhere the
answer it gave on the same inputs is read from tests/golden/reference_results.json.gz.  Record that file (merged with what it
holds) by running the tests where oracle/_ref is built with MPB_RECORD_REFERENCE=1.
"""
from __future__ import annotations

import atexit
import base64
import ctypes as C
import gzip
import hashlib
import json
import os
import subprocess
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORA_DIR = os.path.join(ROOT, "oracle")
REF_SO = os.path.join(ORA_DIR, "_ref", "libref.so")
REF_BIN = os.path.join(ORA_DIR, "_ref", "miniprot")
ORA_SO = os.path.join(ORA_DIR, "liboracle.so")
GOLDEN = os.path.join(ROOT, "tests", "golden")
RECORDED = os.path.join(GOLDEN, "reference_results.json.gz")
# the reference's two bundled test inputs (data)
DPP3_GEN, DPP3_PEP = os.path.join(GOLDEN, "DPP3-hs.gen.fa.gz"), os.path.join(GOLDEN, "DPP3-mm.pep.fa.gz")

_recorded = None
_record = os.environ.get("MPB_RECORD_REFERENCE") == "1"


def _save_recorded():
    with open(RECORDED, "wb") as f, gzip.GzipFile(fileobj=f, mode="wb", mtime=0) as z:
        z.write(json.dumps(_recorded, sort_keys=True, separators=(",", ":")).encode())


def _canon(x):
    """x as plain JSON data (numpy scalars as Python numbers, byte strings and ctypes arrays as their sha256, ctypes structures
    as field dicts), so that a key does not depend on how a value prints."""
    if isinstance(x, (bytes, bytearray, memoryview)):
        return "sha256:" + digest(x)
    if isinstance(x, (bool, np.bool_)):
        return bool(x)
    if isinstance(x, (int, np.integer)):
        return int(x)
    if isinstance(x, (float, np.floating)):
        return float(x)
    if isinstance(x, C.Structure):
        return {f: _canon(getattr(x, f)) for f, _ in x._fields_}
    if isinstance(x, C.Array):
        return _canon(bytes(x))
    if isinstance(x, dict):
        return {str(k): _canon(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_canon(v) for v in x]
    if x is None or isinstance(x, str):
        return x
    raise TypeError(f"no canonical form for {type(x).__name__}")


def reference(kind: str, parts, compute):
    """The reference's answer (JSON data) to one call identified by `kind` and its inputs `parts`: compute() where the reference
    is built -- checked against the answer recorded for the same inputs, if there is one -- else the recorded answer."""
    global _recorded
    key = f"{kind}:" + hashlib.sha256(json.dumps([kind, _canon(list(parts))], sort_keys=True).encode()).hexdigest()[:32]
    if _recorded is None:
        _recorded = json.loads(gzip.open(RECORDED).read()) if os.path.exists(RECORDED) else {}
        if _record:
            atexit.register(_save_recorded)
    if have_ref():
        v = json.loads(json.dumps(compute()))  # the same types as a recorded answer
        if _record:
            _recorded[key] = v
        elif key in _recorded and _recorded[key] != v:
            raise AssertionError(f"the reference now answers this {kind} call ({key}) differently from the answer recorded in "
                                 f"{os.path.relpath(RECORDED, ROOT)}: record it again (MPB_RECORD_REFERENCE=1)")
        return v
    if key not in _recorded:
        raise KeyError(f"no recorded answer of the reference for this {kind} call ({key}): record it where oracle/_ref is built "
                       f"(MPB_RECORD_REFERENCE=1)")
    return _recorded[key]


def digest(b) -> str:
    return hashlib.sha256(bytes(b)).hexdigest()


def file_digest(path: str) -> str:
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 24), b""):
            h.update(blk)
    return h.hexdigest()


def ref_cli(args, g, p, threads=8, index=None) -> dict:
    """md5 and line count of what the reference CLI prints for `args` on genome `g` and proteins `p`; where the reference is run
    here also `out`, `err` and `s`: its stdout, its stderr and its wall time in seconds.  index: an .mpi of `g` for the reference to restore instead of indexing g
    (the index file is part of the reference's contract: tests/test_tables.py::test_index_file_is_byte_identical)."""
    out = {}

    def run():
        t0 = time.perf_counter()
        r = subprocess.run([REF_BIN, f"-t{threads}", *args, index or g, p], check=True, capture_output=True)
        out["out"], out["err"], out["s"] = r.stdout, r.stderr, time.perf_counter() - t0
        return {"md5": hashlib.md5(r.stdout).hexdigest(), "lines": r.stdout.count(b"\n")}

    return dict(reference("cli", (list(args), file_digest(g), file_digest(p)), run), **out)


def _b64(a: np.ndarray) -> str:
    return base64.b64encode(np.ascontiguousarray(a).tobytes()).decode()


def _unb64(s: str, dtype) -> np.ndarray:
    return np.frombuffer(base64.b64decode(s), dtype=dtype).copy()


def build_oracle():
    subprocess.run(["make", "-s", "-C", ORA_DIR, "all"], check=True, stdout=subprocess.DEVNULL)


class NsOpt(C.Structure):  # reference nasw.h:61-71 (== include/nasw_b200.h ns_opt_t)
    _fields_ = [("flag", C.c_int32), ("go", C.c_int32), ("ge", C.c_int32), ("io", C.c_int32), ("fs", C.c_int32),
                ("xdrop", C.c_int32), ("end_bonus", C.c_int32), ("asize", C.c_int32), ("sp", C.c_int32 * 6),
                ("sp_null_bonus", C.c_int32), ("ie_coef", C.c_float), ("sc", C.c_void_p), ("nt4", C.c_void_p),
                ("aa20", C.c_void_p), ("codon", C.c_void_p)]


class NsRst(C.Structure):  # reference nasw.h:73-78
    _fields_ = [("n_cigar", C.c_int32), ("m_cigar", C.c_int32), ("nt_len", C.c_int32), ("aa_len", C.c_int32),
                ("score", C.c_int32), ("cigar", C.POINTER(C.c_uint32))]


class OraTab(C.Structure):
    _fields_ = [("nt4", C.c_void_p), ("aa20", C.c_void_p), ("aa13", C.c_void_p), ("codon", C.c_void_p), ("codon13", C.c_void_p)]


class OraNaswPar(C.Structure):
    _fields_ = [("flag", C.c_int32), ("go", C.c_int32), ("ge", C.c_int32), ("io", C.c_int32), ("fs", C.c_int32),
                ("xdrop", C.c_int32), ("end_bonus", C.c_int32), ("sp", C.c_int32 * 6), ("sp_null_bonus", C.c_int32),
                ("ie_coef", C.c_float), ("mat", C.c_void_p)]


class OraNaswRst(C.Structure):
    _fields_ = [("score", C.c_int32), ("nt_len", C.c_int32), ("aa_len", C.c_int32), ("n_cigar", C.c_int32),
                ("m_cigar", C.c_int32), ("cigar", C.POINTER(C.c_uint32))]


class ChainPar(C.Structure):
    _fields_ = [("max_dist_x", C.c_int32), ("max_dist_y", C.c_int32), ("bw", C.c_int32), ("max_skip", C.c_int32),
                ("max_iter", C.c_int32), ("min_cnt", C.c_int32), ("min_sc", C.c_int32), ("chn_coef_log", C.c_float),
                ("is_spliced", C.c_int32), ("kmer", C.c_int32), ("bbit", C.c_int32)]


_ref = None
_ora = None
_libc = C.CDLL(None)
_libc.free.argtypes = [C.c_void_p]


def have_ref() -> bool:
    return os.path.exists(REF_SO)


def ref():
    global _ref
    if _ref is None:
        _ref = C.CDLL(REF_SO)
        _ref.ref_mp_start()
        _ref.ref_mp_chain.restype = C.c_void_p
        _ref.ref_mp_chain.argtypes = [C.c_int32] * 7 + [C.c_float] + [C.c_int32] * 3 + [C.c_int64, C.c_void_p,
                                                                                       C.POINTER(C.c_int32),
                                                                                       C.POINTER(C.c_void_p), C.c_void_p]
        _ref.ref_kmalloc.restype = C.c_void_p
        _ref.ref_kmalloc.argtypes = [C.c_void_p, C.c_size_t]
        _ref.ref_ns_global_gs16b.argtypes = [C.c_void_p, C.c_char_p, C.c_int32, C.c_char_p, C.c_int32, C.POINTER(NsOpt),
                                             C.c_void_p, C.POINTER(NsRst)]
    return _ref


def ora():
    global _ora
    if _ora is None:
        if not os.path.exists(ORA_SO):
            build_oracle()
        _ora = C.CDLL(ORA_SO)
        _ora.ora_chain.restype = C.c_void_p
        _ora.ora_chain.argtypes = [C.POINTER(ChainPar), C.c_int64, C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_void_p)]
        _ora.ora_seed_anchors.restype = C.c_void_p
        _ora.ora_refine.restype = C.c_void_p
        _ora.ora_hash32_mask.restype = C.c_uint32
        _ora.ora_hash32_mask.argtypes = [C.c_uint32, C.c_uint32]
        _ora.ora_sketch_nt4.restype = C.c_int64
    return _ora


_TAB_SIZES = (("nt4", 256), ("aa20", 256), ("aa13", 256), ("codon", 64), ("codon13", 64))
_ref_tab = None


def ref_tables() -> OraTab:
    """Oracle table bundle with a copy of the REFERENCE's tables (after ref_mp_start())."""
    global _ref_tab
    if _ref_tab is None:
        tabs = reference("tables", (), lambda: {f: _b64(np.ctypeslib.as_array((C.c_uint8 * n).in_dll(ref(), "ref_ns_tab_" + f)))
                                                for f, n in _TAB_SIZES})
        arr = [_unb64(tabs[f], np.uint8) for f, _ in _TAB_SIZES]
        _ref_tab = (tables_from_arrays(*arr), arr)
    return _ref_tab[0]


def tables_from_arrays(nt4, aa20, aa13, codon, codon13):
    """Oracle table bundle from numpy uint8 arrays (kept alive by the caller)."""
    t = OraTab()
    t.nt4, t.aa20, t.aa13, t.codon, t.codon13 = (a.ctypes.data for a in (nt4, aa20, aa13, codon, codon13))
    return t


DEFAULT_NASW = dict(go=11, ge=1, io=29, fs=23, xdrop=100, end_bonus=5, sp=(8, 15, 21, 30, 0, 0), sp_null_bonus=-7,
                    ie_coef=0.5)


def default_mat() -> np.ndarray:
    """BLOSUM62 22x22 with the miniprot stop-codon row (options.c:87-88), the reference's."""
    def compute():
        m = np.ctypeslib.as_array((C.c_int8 * 484).in_dll(ref(), "ref_ns_mat_blosum62")).copy()
        ref().ref_ns_set_stop_sc(22, m.ctypes.data_as(C.c_void_p), 23)
        return _b64(m)

    return _unb64(reference("default_mat", (), compute), np.int8)


def ref_set_stop_sc(mat: np.ndarray, sc: int) -> None:
    """The reference's ns_set_stop_sc(22, mat, sc) (-C, options.c:87-88), in place."""
    def compute():
        m = mat.copy()
        ref().ref_ns_set_stop_sc(22, m.ctypes.data_as(C.c_void_p), sc)
        return _b64(m)

    mat[:] = _unb64(reference("set_stop_sc", (mat.tobytes(), sc), compute), np.int8)


def ref_nasw(nt: np.ndarray, aa: bytes, flag: int, mat: np.ndarray, par: dict, ss=None):
    def compute():
        r = ref()
        o = NsOpt()
        r.ref_ns_opt_init(C.byref(o))
        for k in ("go", "ge", "io", "fs", "xdrop", "end_bonus", "sp_null_bonus", "ie_coef"):
            setattr(o, k, par[k])
        for i in range(6):
            o.sp[i] = par["sp"][i]
        o.flag = flag
        o.sc = mat.ctypes.data
        rst = NsRst()
        ssp = ss.ctypes.data_as(C.c_void_p) if ss is not None else None
        r.ref_ns_global_gs16b(None, nt.tobytes(), len(nt), aa, len(aa), C.byref(o), ssp, C.byref(rst))
        cig = [rst.cigar[i] for i in range(rst.n_cigar)]
        if rst.n_cigar:
            _libc.free(rst.cigar)
        return [rst.score, rst.nt_len, rst.aa_len, cig]

    parts = (np.ascontiguousarray(nt, dtype=np.uint8).tobytes(), bytes(aa), flag, mat.tobytes(), par,
             None if ss is None else np.ascontiguousarray(ss, dtype=np.uint8).tobytes())
    score, nt_len, aa_len, cig = reference("nasw", parts, compute)
    return score, nt_len, aa_len, cig


def ref_sort128x(z: np.ndarray) -> str:
    """sha256 of what the reference's radix_sort_mp128x makes of the (n, 2) uint64 array z."""
    def compute():
        a = z.copy()
        ref().ref_radix_sort_mp128x(a.ctypes.data_as(C.c_void_p), C.c_void_p(a.ctypes.data + 16 * len(a)))
        return digest(a.tobytes())

    return reference("sort128x", (z.tobytes(),), compute)


class _Mp64(C.Structure):  # mp64_v
    _fields_ = [("n", C.c_int32), ("m", C.c_int32), ("a", C.POINTER(C.c_uint64))]


def _take_mp64(v: _Mp64):
    a = np.ctypeslib.as_array(v.a, shape=(v.n,)).copy() if v.n else np.zeros(0, np.uint64)
    if v.a:
        _libc.free(v.a)
    return [v.n, digest(a.tobytes())]


def ref_sketch_prot(seq: bytes, k: int, m: int):
    """(n, sha256 of the n uint64s) of the reference's mp_sketch_prot."""
    def compute():
        v = _Mp64()
        ref().ref_mp_sketch_prot(None, seq, len(seq), k, m, C.byref(v))
        return _take_mp64(v)

    return tuple(reference("sketch_prot", (seq, k, m), compute))


def ref_sketch_nt4(nt: np.ndarray, k: int, m: int, bbit: int, boff: int):
    """(n, sha256 of the n uint64s) of the reference's mp_sketch_nt4 (min_aa_len 30)."""
    def compute():
        v = _Mp64()
        ref().ref_mp_sketch_nt4(None, nt.ctypes.data_as(C.c_void_p), C.c_int64(len(nt)), 30, k, m, bbit, C.c_int64(boff), C.byref(v))
        return _take_mp64(v)

    return tuple(reference("sketch_nt4", (nt.tobytes(), k, m, bbit, boff), compute))


def ora_nasw(tab: OraTab, nt: np.ndarray, aa: bytes, flag: int, mat: np.ndarray, par: dict, ss=None):
    o = ora()
    p = OraNaswPar()
    for k in ("go", "ge", "io", "fs", "xdrop", "end_bonus", "sp_null_bonus", "ie_coef"):
        setattr(p, k, par[k])
    for i in range(6):
        p.sp[i] = par["sp"][i]
    p.flag = flag
    p.mat = mat.ctypes.data
    rst = OraNaswRst()
    nt = np.ascontiguousarray(nt, dtype=np.uint8)
    ssp = ss.ctypes.data_as(C.c_void_p) if ss is not None else None
    o.ora_nasw(C.byref(tab), C.byref(p), nt.ctypes.data_as(C.c_void_p), len(nt), aa, len(aa), ssp, C.byref(rst))
    cig = [rst.cigar[i] for i in range(rst.n_cigar)]
    if rst.n_cigar:
        _libc.free(rst.cigar)
    return rst.score, rst.nt_len, rst.aa_len, cig


# ------------------------------------------------------------------ random problem generators

_AA = "ARNDCQEGHILKMFPSTWYV"
_STD = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"
_T2A = {"T": 3, "C": 1, "A": 0, "G": 2}
_AA2COD = {}
for _i, _a in enumerate(_STD):
    _c = ("TCAG"[_i >> 4], "TCAG"[(_i >> 2) & 3], "TCAG"[_i & 3])
    _AA2COD.setdefault(_a, []).append([_T2A[x] for x in _c])


def random_dp_problem(rng: np.random.Generator, al_max=60, intron_max=400, p_sub=0.2, p_indel=0.03, p_fs=0.02, p_n=0.002,
                      flank=30):
    """A protein and a nucleotide string (codes 0..4) that encodes a mutated, intron-interrupted copy of it."""
    al = int(rng.integers(1, al_max + 1))
    prot = [int(x) for x in rng.integers(0, 20, size=al)]
    nt = []
    nt += [int(x) for x in rng.integers(0, 4, size=int(rng.integers(0, flank + 1)))]
    for a in prot:
        r = rng.random()
        if r < p_indel / 2:
            continue  # residue missing from the genome (insertion in the protein)
        if r < p_indel:
            extra = _AA2COD[_AA[int(rng.integers(0, 20))]]
            nt += extra[int(rng.integers(0, len(extra)))]  # extra codon (deletion)
        aa = _AA[a] if rng.random() >= p_sub else _AA[int(rng.integers(0, 20))]
        if rng.random() < 0.01:
            aa = "*"
        cods = _AA2COD[aa]
        cod = list(cods[int(rng.integers(0, len(cods)))])
        if rng.random() < p_fs:
            if rng.random() < 0.5:
                cod.pop(int(rng.integers(0, 3)))
            else:
                cod.insert(int(rng.integers(0, 3)), int(rng.integers(0, 4)))
        if rng.random() < 0.08 and intron_max > 0:  # intron at a random phase inside this codon
            ph = int(rng.integers(0, len(cod) + 1))
            il = int(rng.integers(20, intron_max + 1))
            body = [int(x) for x in rng.integers(0, 4, size=il)]
            if rng.random() < 0.9:
                body[0:2] = [2, 3]
                body[2] = int(rng.choice([0, 2]))
                body[-3] = int(rng.choice([1, 3]))
                body[-2:] = [0, 2]
            cod = cod[:ph] + body + cod[ph:]
        nt += cod
    nt += [int(x) for x in rng.integers(0, 4, size=int(rng.integers(0, flank + 1)))]
    nt = np.array(nt, dtype=np.uint8)
    if len(nt) and p_n > 0:
        nt[rng.random(len(nt)) < p_n] = 4
    aa = "".join(_AA[a] for a in prot)
    if rng.random() < 0.1 and al > 2:
        k = int(rng.integers(0, al))
        aa = aa[:k] + "X" + aa[k + 1:]
    return nt, aa.encode()


def random_chain_problem(rng: np.random.Generator, n: int, mode: str):
    """Sorted anchors for the three mp_chain call regimes: 'pre', 'main' (block ids) and 'refine' (base resolution)."""
    if mode in ("pre", "main"):
        nb = max(4, n // 3)
        x = np.sort(rng.integers(1000, 1000 + nb, size=n)).astype(np.uint64)
        base = rng.integers(5, 400, size=n)
        # plant collinear runs: qpos follows block id * 85 (256/3) within clusters
        y = ((x.astype(np.int64) - 1000) * 85 % 380 + rng.integers(0, 40, size=n) + 5).astype(np.uint64)
        y = np.where(rng.random(n) < 0.3, base.astype(np.uint64), y)
    else:
        x = np.sort(rng.integers(14, 14 + 6 * n + 50, size=n)).astype(np.uint64)
        y = (x.astype(np.int64) // 3 + rng.integers(-3, 4, size=n)).clip(4, 2000).astype(np.uint64)
        y = np.where(rng.random(n) < 0.2, rng.integers(4, 500, size=n).astype(np.uint64), y)
    a = np.unique((x << np.uint64(32)) | y)
    return np.ascontiguousarray(a, dtype=np.uint64)


CHAIN_MODES = {
    "pre": dict(max_dist_x=256, max_dist_y=256, bw=256, max_skip=25, max_iter=1000000, min_cnt=2, min_sc=0,
                chn_coef_log=0.75, is_spliced=1, kmer=6, bbit=8),
    "main": dict(max_dist_x=200000, max_dist_y=1000, bw=200000, max_skip=25, max_iter=1000000, min_cnt=3, min_sc=0,
                 chn_coef_log=0.75, is_spliced=1, kmer=6, bbit=8),
    "refine": dict(max_dist_x=200000, max_dist_y=1000, bw=200000, max_skip=25, max_iter=1000000, min_cnt=3, min_sc=0,
                   chn_coef_log=0.75, is_spliced=1, kmer=5, bbit=0),
}


def chain_par(mode: str, **over) -> ChainPar:
    d = dict(CHAIN_MODES[mode])
    d.update(over)
    return ChainPar(**d)


def ref_chain(par: ChainPar, a: np.ndarray):
    def compute():
        r = ref()
        n = len(a)
        buf = r.ref_kmalloc(None, max(8 * n, 8))  # mp_chain frees its input
        C.memmove(buf, a.ctypes.data, 8 * n)
        n_u = C.c_int32(0)
        u = C.c_void_p(0)
        b = r.ref_mp_chain(par.max_dist_x, par.max_dist_y, par.bw, par.max_skip, par.max_iter, par.min_cnt, par.min_sc,
                           par.chn_coef_log, par.is_spliced, par.kmer, par.bbit, n, buf, C.byref(n_u), C.byref(u), None)
        return [_b64(x) for x in _take_chain(n_u.value, u.value, b)]

    u, b = reference("chain", (par, a.tobytes()), compute)
    return _unb64(u, np.uint64), _unb64(b, np.uint64)


def _take_chain(n_u, u_ptr, b_ptr):
    if n_u == 0:
        return np.zeros(0, np.uint64), np.zeros(0, np.uint64)
    u = np.ctypeslib.as_array(C.cast(u_ptr, C.POINTER(C.c_uint64)), shape=(n_u,)).copy()
    nb = int((u & np.uint64(0xffffffff)).sum())
    b = np.ctypeslib.as_array(C.cast(b_ptr, C.POINTER(C.c_uint64)), shape=(nb,)).copy()
    _libc.free(u_ptr)
    _libc.free(b_ptr)
    return u, b


def ora_chain(par: ChainPar, a: np.ndarray):
    o = ora()
    n_u = C.c_int32(0)
    u = C.c_void_p(0)
    b = o.ora_chain(C.byref(par), len(a), a.ctypes.data_as(C.c_void_p), C.byref(n_u), C.byref(u))
    return _take_chain(n_u.value, u.value, b)
