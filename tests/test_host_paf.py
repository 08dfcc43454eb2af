"""CPU: the product's HOST pipeline (region bookkeeping, alignment planner, statistics, PAF writer, index builder) with
the C oracle plugged in as stage backend must reproduce the reference's PAF byte for byte (golden fixtures)."""
import ctypes as C
import os

import pytest

import build_hostcheck
import oracle_lib as ol
from miniprot_b200 import synth

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")


@pytest.fixture(scope="module")
def hc():
    lib = C.CDLL(build_hostcheck.build())
    lib.hc_map_file.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_uint32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int64]
    return lib


def run(hc, g, p, out, flag=0, max_intron=0, auto=0, sp=-1, mini_batch=0):
    assert hc.hc_map_file(g.encode(), p.encode(), out.encode(), flag, max_intron, auto, sp, 4, mini_batch) == 0
    return open(out, "rb").read()


@pytest.mark.parametrize("name,kw", [("DPP3_default", {}), ("DPP3_j2", dict(sp=2)), ("DPP3_G2k", dict(max_intron=2000))])
def test_dpp3_golden(hc, tmp_path, name, kw):
    got = run(hc, ol.DPP3_GEN, ol.DPP3_PEP, str(tmp_path / "o.paf"), **kw)
    assert got == open(os.path.join(GOLD, name + ".paf"), "rb").read()


@pytest.mark.parametrize("cfg", ["tiny", "tiny5"])
def test_synthetic_golden(hc, tmp_path, cfg, monkeypatch):
    g, p = synth.generate(synth.CONFIGS[cfg], str(tmp_path))
    want = open(os.path.join(GOLD, cfg + ".paf"), "rb").read()
    assert run(hc, g, p, str(tmp_path / "o.paf")) == want
    # batch boundaries must not matter (SURVEY 8b determinism contract): 3 proteins per mini-batch
    assert run(hc, g, p, str(tmp_path / "o2.paf"), mini_batch=1200) == want
    # ... nor whether the three steps of the file driver (read / map / write, map.c:273-343) overlap or run one after another
    monkeypatch.setenv("MPB_FILE_PIPELINE", "0")
    assert run(hc, g, p, str(tmp_path / "o3.paf"), mini_batch=1200) == want
    assert run(hc, g, p, str(tmp_path / "o4.paf"), mini_batch=1) == want  # one protein per mini-batch
    monkeypatch.delenv("MPB_FILE_PIPELINE")
    assert run(hc, g, p, str(tmp_path / "o5.paf"), mini_batch=1) == want


FORMATS = {"gff": (0x8, None), "gtf": (0x20, None), "aln": (0x80, None), "trans": (0x100 | 0x4, None), "gff_only": (0x8 | 0x10, "#")}


@pytest.mark.parametrize("fmt", sorted(FORMATS))
def test_other_output_formats_golden(hc, tmp_path, fmt, monkeypatch):
    """GFF3 / GTF / --aln / --trans / --gff-only with --gff-delim (format.c:189-452) against the reference's output: the set
    with every CIGAR operation (tiny5) and the bundled DPP3 pair (md5s of SURVEY App. D)."""
    import gzip

    flag, delim = FORMATS[fmt]
    if delim:
        monkeypatch.setenv("HC_GFF_DELIM", delim)
    g, p = synth.generate(synth.CONFIGS["tiny5"], str(tmp_path))
    gold = os.path.join(GOLD, f"tiny5_{fmt}.txt")
    want = gzip.open(gold + ".gz", "rb").read() if os.path.exists(gold + ".gz") else open(gold, "rb").read()
    assert run(hc, g, p, str(tmp_path / "o.txt"), flag=flag) == want
    assert run(hc, g, p, str(tmp_path / "o2.txt"), flag=flag, mini_batch=1200) == want  # the hit counter runs across mini-batches
    got = run(hc, ol.DPP3_GEN, ol.DPP3_PEP, str(tmp_path / "d.txt"), flag=flag)
    assert got == open(os.path.join(GOLD, f"DPP3_{fmt}.txt"), "rb").read()


@pytest.mark.parametrize("extra", [0, 1, 2, 3, 4])
def test_hit_abutting_the_contig_end(hc, tmp_path, extra, capfd):
    """A gene whose coding sequence stops `extra` bases before the contig end while the protein goes on: with fewer than 3 bases left
    there is nothing to extend into (the reference stops at an assertion there, nasw-sse.c:443); the hit must simply end at its last
    pinned anchor -- no right extension planned, no `inconsistent CIGAR` drop (align.cpp plan(): has_right)."""
    import numpy as np

    rng = np.random.default_rng(17 + extra)
    aa2cod = {}
    std = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"
    for i, a in enumerate(std):
        aa2cod.setdefault(a, []).append("TCAG"[i >> 4] + "TCAG"[(i >> 2) & 3] + "TCAG"[i & 3])
    prot = "".join("ARNDCQEGHILKMFPSTWYV"[x] for x in rng.integers(0, 20, 160))
    cds = "".join(aa2cod[a][int(rng.integers(0, len(aa2cod[a])))] for a in prot[:120])  # the genome encodes residues 0..119 only
    ctg = "".join("ACGT"[x] for x in rng.integers(0, 4, 5000)) + cds + "".join("ACGT"[x] for x in rng.integers(0, 4, extra))
    g, p = str(tmp_path / "g.fa"), str(tmp_path / "p.faa")
    open(g, "w").write(">ctg\n" + ctg + "\n")
    open(p, "w").write(">prot\n" + prot + "\n")
    paf = run(hc, g, p, str(tmp_path / "o.paf")).decode()
    err = capfd.readouterr().err
    assert "inconsistent CIGAR" not in err, err
    rows = [l.split("\t") for l in paf.splitlines()]
    assert len(rows) >= 1 and rows[0][0] == "prot" and rows[0][5] == "ctg"
    assert int(rows[0][8]) <= len(ctg) and int(rows[0][8]) >= len(ctg) - extra - 30  # the hit reaches the end of the coding sequence
    assert int(rows[0][3]) >= 110 and int(rows[0][3]) <= 121                         # ... and covers the encoded residues only
