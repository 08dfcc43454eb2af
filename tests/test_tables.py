"""CPU: the product library loads, exports every symbol of include/*.h, and its tables / defaults equal the reference's."""
import ctypes as C
import json
import os
import re

import pytest

import miniprot_b200 as mp
import oracle_lib as ol

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    if not os.path.exists(mp.LIB_PATH):
        mp.build()
    return mp.lib()


def test_exports_every_declared_symbol(L):
    names = set()
    for h in ("miniprot_b200.h", "nasw_b200.h"):
        src = open(os.path.join(ROOT, "include", h)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        names |= set(re.findall(r"\b((?:mp|mpb|ns)_[a-z0-9_]+)\s*\(", src))
    names -= {"mp_tbuf_s"}
    missing = [n for n in sorted(names) if not hasattr(L, n)]
    assert not missing, missing
    for g in ("mp_verbose", "mp_dbg_flag", "ns_tab_nt4", "ns_tab_aa20", "ns_tab_aa13", "ns_tab_codon", "ns_tab_codon13", "ns_tab_a2r",
              "ns_mat_blosum62", "ns_tab_nt_i2c", "ns_tab_aa_i2c"):
        C.c_uint8.in_dll(L, g)


TABLES = (("ns_tab_nt4", 256), ("ns_tab_aa20", 256), ("ns_tab_aa13", 256), ("ns_tab_codon", 64), ("ns_tab_codon13", 64), ("ns_tab_a2r", 22))
GSIZES = (1000, 10**8, 3 * 10**9, 10**11)


def _opt_fields(o):
    return {f: (bytes(v).hex() if f == "mat" else v.decode() if isinstance(v, bytes) else v) for f, _ in o._fields_ for v in [getattr(o, f)]}


def _defaults(L, pre=""):
    """Translation tables of several genetic codes, option defaults and -I's max intron, through library L (symbols prefixed `pre`)."""
    fn = lambda name: getattr(L, pre + name)  # noqa: E731
    d = {"tables": {}}
    for code in (1, 2, 4, 11, 33):
        assert fn("ns_make_tables")(code) == 0
        d["tables"][str(code)] = {name: bytes((C.c_uint8 * n).in_dll(L, pre + name)).hex() for name, n in TABLES}
    d["make_tables_7"] = fn("ns_make_tables")(7)
    fn("ns_make_tables")(1)
    d["blosum62"] = bytes((C.c_int8 * 484).in_dll(L, pre + "ns_mat_blosum62")).hex()
    mo, io, no = mp.MapOpt(), mp.IdxOpt(), mp.NsOpt()
    fn("mp_mapopt_init")(C.byref(mo))
    fn("mp_idxopt_init")(C.byref(io))
    fn("ns_opt_init")(C.byref(no))
    d["mapopt"], d["idxopt"] = _opt_fields(mo), bytes(io).hex()
    d["nsopt"] = {f: getattr(no, f) for f in ("go", "ge", "io", "fs", "xdrop", "end_bonus", "asize", "sp_null_bonus", "ie_coef")}
    d["nsopt"]["sp"] = list(no.sp)
    if pre:
        fn("mp_mapopt_set_max_intron").argtypes = [C.c_void_p, C.c_int64]
    C.c_int32.in_dll(L, pre + "mp_verbose").value = 1
    d["max_intron_bw"] = []
    for gsize in GSIZES:
        fn("mp_mapopt_set_max_intron")(C.addressof(mo) if pre else C.byref(mo), gsize)
        d["max_intron_bw"].append([mo.max_intron, mo.bw])
    return d


def test_tables_and_defaults_equal_reference(L):
    ours = json.loads(json.dumps(_defaults(L)))
    want = ol.reference("defaults", (), lambda: _defaults(ol.ref(), "ref_"))
    for code in want["tables"]:
        for name, _ in TABLES:
            assert ours["tables"][code][name] == want["tables"][code][name], (code, name)
    assert ours["make_tables_7"] == want["make_tables_7"] == -2
    for k in ("blosum62", "idxopt", "nsopt", "max_intron_bw"):
        assert ours[k] == want[k], k
    for f in want["mapopt"]:
        assert ours["mapopt"][f] == want["mapopt"][f], f


def test_index_file_is_byte_identical(L, tmp_path):
    """mp_idx_build + mp_idx_dump vs the reference's -d output on a small synthetic genome (ki/kb order is part of the contract)."""
    import subprocess
    from miniprot_b200 import synth

    g, _ = synth.generate(synth.CONFIGS["tiny"], str(tmp_path))
    ours, ref = str(tmp_path / "ours.mpi"), str(tmp_path / "ref.mpi")
    mi = mp.idx_load(g, 4)
    assert L.mp_idx_dump(ours.encode(), mi) == 0
    L.mp_idx_destroy(mi)

    def ref_dump():
        subprocess.run([ol.REF_BIN, "-t4", "-d", ref, g], check=True, stderr=subprocess.DEVNULL)
        return ol.file_digest(ref)

    assert ol.file_digest(ours) == ol.reference("idx_dump", (ol.file_digest(g),), ref_dump)
    mi2 = L.mp_idx_restore((ref if os.path.exists(ref) else ours).encode())
    assert mi2 and mi2.contents.n_kb > 0
    L.mp_idx_destroy(mi2)


def test_no_gpu_means_loud_failure(L):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError):
        mp.Context(0)


class Spsc(C.Structure):
    _fields_ = [("n", C.c_uint32), ("m", C.c_uint32), ("a", C.POINTER(C.c_uint64))]


def _spsc(L, pre, g, sp):
    """(io, io_end) after mp_set_spsc and the per-strand arrays (length, sha256) it leaves in the index, for keep_io 0 and 1."""
    fn = getattr(L, pre + "mp_idx_load")
    fn.restype = C.POINTER(mp.Idx)
    mi = fn(g.encode(), C.byref(mp.idxopt()), 4)
    out = []
    for keep_io in (0, 1):
        mo = mp.mapopt()
        getattr(L, pre + "mp_set_spsc")(sp.encode(), mi, C.byref(mo), keep_io)
        sa = C.cast(mi.contents.nt.contents.spsc, C.POINTER(Spsc))
        arrays = [[sa[j].n, ol.digest(C.string_at(sa[j].a, 8 * sa[j].n) if sa[j].n else b"")] for j in range(2 * mi.contents.nt.contents.n_ctg)]
        out.append([[mo.io, mo.io_end], arrays])
    getattr(L, pre + "mp_idx_destroy")(mi)
    return out


def test_splice_score_reader_equals_reference(L, tmp_path):
    """mp_set_spsc / mp_ntseq_read_spsc (index.c:239-248, ntseq.c:234-296): option side effects and the sorted per-strand arrays."""
    from miniprot_b200 import synth
    g, _ = synth.generate(synth.CONFIGS["tiny"], str(tmp_path))
    sp = synth.make_spsc(g, str(tmp_path / "t.spsc"), seed=3, p_site=0.2, p_noise=0.001)
    ours = json.loads(json.dumps(_spsc(L, "", g, sp)))
    want = ol.reference("spsc", (ol.file_digest(g), ol.file_digest(sp)), lambda: _spsc(ol.ref(), "ref_", g, sp))
    for keep_io, ((io, arrays), (wio, warrays)) in enumerate(zip(ours, want)):
        assert io == wio == ([29, 19] if keep_io else [39, 29])
        assert len(arrays) == len(warrays)
        for j, (a, w) in enumerate(zip(arrays, warrays)):
            assert a == w, j
        assert sum(n for n, _ in warrays) > 1000


def test_build_record_matches_the_loaded_library():
    """build() records what the library was compiled from (BUILD_INFO.json); bench.py and smoke() report it, so a stale or foreign
    .so would show (so_is_that_build / sources_unchanged_since false)."""
    import os

    import miniprot_b200 as mp

    if not os.path.exists(mp.BUILD_INFO):
        import pytest

        pytest.skip("library was built outside miniprot_b200.build()")
    bi = mp.build_info()
    assert "error" not in bi and bi["so_is_that_build"] and bi["sources_unchanged_since"], bi
    assert "compute_100a" in bi["arch"] and len(bi["source_sha256"]) == 64
