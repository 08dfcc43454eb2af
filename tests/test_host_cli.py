"""CPU: the reference's UNMODIFIED command-line front end (main.c, compiled where it lies) linked against the product's HOST sources
with the C oracle as stage backend (tests/_build/libhostcheck.so) must print what the reference binary prints, byte for byte, under
random command lines -- scoring, chaining and output options, every output format, --spsc, index dump / restore (crosswise) -- on
random synthetic inputs that include awkward query records.  A fixed-seed slice of tools/fuzz_cli.py (which runs open-ended).
Needs oracle/_ref/miniprot and oracle/_ref/miniprot_hostcheck_cli, which build() makes where the reference sources are present."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import fuzz_cli  # noqa: E402

pytestmark = pytest.mark.skipif(not (os.path.exists(fuzz_cli.CLI) and os.path.exists(fuzz_cli.REF_BIN)),
                                reason="needs oracle/_ref/miniprot and oracle/_ref/miniprot_hostcheck_cli (oracle/Makefile)")


@pytest.mark.parametrize("seed", [101, 202])
def test_random_command_lines_match_the_reference_binary(seed, tmp_path):
    n, bad = fuzz_cli.fuzz(seed, 30, str(tmp_path))
    assert n == 30 and bad == 0
