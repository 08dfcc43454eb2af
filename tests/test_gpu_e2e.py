"""GPU end-to-end parity: FASTA proteins -> PAF through mpb_map_file (all stages on the GPU) must be byte-identical to
the reference CLI (oracle/_ref/miniprot run on this box, or its recorded output digest) and to the committed golden PAFs."""
import hashlib
import os
import subprocess

import pytest

import miniprot_b200 as mp
import oracle_lib as ol
from miniprot_b200 import synth

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")


@pytest.fixture(scope="module")
def ctx():
    c = mp.Context(0)
    yield c
    c.close()


def gpu_paf(ctx, g, p, out, **over):
    mi = mp.idx_load(g, 8)
    mo = mp.mapopt(**{k: v for k, v in over.items() if k != "auto_intron"})
    if over.get("auto_intron"):
        mp.lib().mp_mapopt_set_max_intron(mo, mi.contents.nt.contents.l_seq)
    mp.map_file(ctx, mi, p, out, mo)
    mp.lib().mp_idx_destroy(mi)
    return open(out, "rb").read()


def test_dpp3(ctx, tmp_path):
    g, p = ol.DPP3_GEN, ol.DPP3_PEP
    assert gpu_paf(ctx, g, p, str(tmp_path / "o.paf")) == open(os.path.join(GOLD, "DPP3_default.paf"), "rb").read()
    assert gpu_paf(ctx, g, p, str(tmp_path / "o.paf"), sp_model=2) == open(os.path.join(GOLD, "DPP3_j2.paf"), "rb").read()
    assert gpu_paf(ctx, g, p, str(tmp_path / "o.paf"), max_intron=2000, bw=2000) == open(os.path.join(GOLD, "DPP3_G2k.paf"), "rb").read()


@pytest.mark.parametrize("cfg", ["tiny", "tiny5"])
def test_tiny_golden(ctx, tmp_path, cfg):
    g, p = synth.generate(synth.CONFIGS[cfg], str(tmp_path))
    want = open(os.path.join(GOLD, cfg + ".paf"), "rb").read()
    assert gpu_paf(ctx, g, p, str(tmp_path / "o.paf")) == want
    assert gpu_paf(ctx, g, p, str(tmp_path / "o2.paf"), mini_batch_size=1200) == want  # batch boundaries do not matter


@pytest.mark.parametrize("cfg,args,over", [("small", (), {}), ("small5", (), {}), ("small", ("-I",), dict(auto_intron=1)),
                                           ("small5", ("-G", "20k", "-e", "2k"), dict(max_intron=20000, bw=20000, max_ext=2000))])
def test_small_vs_reference_cli(ctx, tmp_path, cfg, args, over):
    g, p = synth.generate(synth.CONFIGS[cfg], str(tmp_path))
    got = gpu_paf(ctx, g, p, str(tmp_path / "o.paf"), **over)
    want = ol.ref_cli(args, g, p)
    if hashlib.md5(got).hexdigest() != want["md5"]:
        a = got.decode().splitlines()
        diff = [(x[:200], y[:200]) for x, y in zip(a, want["out"].decode().splitlines()) if x != y][:3] if "out" in want else "-"
        pytest.fail(f"{cfg} {args}: {len(a)} vs {want['lines']} lines; first diffs: {diff}")


def test_index_loaded_straight_into_hbm(ctx, tmp_path):
    """mpb_idx_load_device: the .mpi file goes to the device through pinned staging buffers, the host keeps no ki / kb
    (SURVEY 8f #3); mapping with it gives the golden PAF, and an index written by the reference CLI loads the same way."""
    g, p = synth.generate(synth.CONFIGS["tiny"], str(tmp_path))
    want = open(os.path.join(GOLD, "tiny.paf"), "rb").read()
    L = mp.lib()
    mi0 = mp.idx_load(g, 4)
    ours = str(tmp_path / "ours.mpi")
    assert L.mp_idx_dump(ours.encode(), mi0) == 0
    L.mp_idx_destroy(mi0)
    files = [ours]
    if os.path.exists(ol.REF_BIN):
        ref = str(tmp_path / "ref.mpi")
        subprocess.run([ol.REF_BIN, "-t4", "-d", ref, g], check=True, capture_output=True)
        files.append(ref)
    for f in files:
        mi = mp.idx_load_device(ctx, f)
        assert not mi.contents.ki and not mi.contents.kb
        mp.map_file(ctx, mi, p, str(tmp_path / "o.paf"))
        L.mp_idx_destroy(mi)
        assert open(str(tmp_path / "o.paf"), "rb").read() == want
