"""GPU parity on the shapes of BASELINE.json's configurations (SURVEY 8d): the whole path (FASTA proteins -> PAF through
mpb_map_file) against the reference CLI (run on the same box, or its recorded output digest), byte for byte.

  C5   100 Mbp, 1000 proteins at 60 % identity with 2 % frameshifts (full size): every scoring branch / CIGAR operation
  C4s  the long-intron stress shape (one 50-150 kbp intron per gene, 400 kbp slots) under the -G x -e sweep
  C3s  the 3 Gbp / -I shape cut down to 1 Gbp: ~48 k anchors per protein (the large chaining class), bw = max_intron from
       the genome size, DP problems of up to 190 k rows
The generators, the option handling and the comparison live in tools/parity.py (also used for the measurements)."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import oracle_lib as ol  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def run(tmp_path_factory):
    import miniprot_b200 as mp
    import parity

    ctx = mp.Context(0)
    base = os.environ.get("MPB_BENCH_DIR", str(tmp_path_factory.mktemp("cfg")))

    def go(cfg, opts):
        rows = parity.run_config(cfg, opts, os.path.join(base, cfg), min(os.cpu_count() or 8, 128), ctx=ctx)
        for r in rows:
            assert r["identical"], f"{cfg} {r['opt']!r}: PAF differs from the reference ({r['paf_lines']} vs {r['ref_lines']} lines): {r.get('first_diffs')}"
        return rows

    yield go
    ctx.close()


def test_c5_full_size(run):
    rows = run("C5", [""])
    assert rows[0]["paf_lines"] > 500


def test_c4_long_intron_sweep(run):
    run("C4s", ["-G 50k -e 2k", "-G 50k -e 50k", "-G 200k -e 2k", "-G 200k -e 50k"])


def test_c3_shape_auto_intron(run):
    rows = run("C3s", ["-I"])
    assert rows[0]["anchors_per_protein"] > 16384  # every pre-chain problem is in the largest chaining class
