"""Differential fuzzing of the HOST side of the product under arbitrary command lines, on the CPU (no GPU needed): the reference's
UNMODIFIED main.c linked against tests/_build/libhostcheck.so (the product's host sources -- options, index builder, .mpi I/O, hit
bookkeeping, alignment planner, statistics, all output formats -- with the C oracle as stage backend) against the reference binary
oracle/_ref/miniprot, same random options, same random synthetic inputs; stdout must be byte-identical.
Needs oracle/_ref (the reference binary and the CLI, built by oracle/Makefile where the reference sources are present).  Test
infrastructure, not part of the product.

usage: python tools/fuzz_cli.py [seed] [n_iterations] [workdir]"""
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import build_hostcheck  # noqa: E402
from miniprot_b200 import synth  # noqa: E402

REF_BIN = os.path.join(ROOT, "oracle", "_ref", "miniprot")
CLI = os.path.join(ROOT, "oracle", "_ref", "miniprot_hostcheck_cli")  # compiled reference source: output under oracle/_ref like the other reference builds


def build_cli():
    """oracle/_ref/miniprot_hostcheck_cli = reference main.c (compiled where it lies) + tests/_build/libhostcheck.so; the recipe is
    oracle/Makefile (target hostcheck_cli, made by __graft_entry__.build() where the reference sources are present; with
    MPB_REFERENCE=<reference source directory> it is remade here).  None if it has not been built."""
    build_hostcheck.build()
    if os.environ.get("MPB_REFERENCE"):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "hostcheck_cli", "REF=" + os.environ["MPB_REFERENCE"]], check=True)
    return CLI if os.path.exists(CLI) else None


def random_inputs(rng, d):
    spec = synth.SynthSpec(genome_len=int(rng.choice([300_000, 600_000, 1_200_000])), n_genes=int(rng.integers(4, 16)),
                           identity=float(rng.choice([0.95, 0.8, 0.6])), lmax=int(rng.choice([300, 2000, 8000])), seed=int(rng.integers(1, 1 << 30)),
                           ctg_len=int(rng.choice([100_000, 250_000, 2_000_000])), fs_per_base=float(rng.choice([0.0, 0.0, 0.0067])),
                           min_exons=int(rng.choice([1, 3])), max_exons=int(rng.choice([3, 8])))
    g, p = synth.generate(spec, d)
    if rng.random() < 0.6:  # paralogs: diverged copies of random segments (whole or partial genes, either strand) elsewhere in the genome
        comp = bytes.maketrans(b"ACGT", b"TGCA")
        recs = [r.split("\n", 1) for r in open(g).read().split(">")[1:]]
        seqs = [bytearray(r[1].replace("\n", "").encode()) for r in recs]
        for _ in range(int(rng.integers(2, 12))):
            a, b = int(rng.integers(0, len(seqs))), int(rng.integers(0, len(seqs)))
            ln = int(rng.integers(1500, 20000))
            if len(seqs[a]) <= ln + 10 or len(seqs[b]) <= ln + 10:
                continue
            s0, t0 = int(rng.integers(0, len(seqs[a]) - ln)), int(rng.integers(0, len(seqs[b]) - ln))
            seg = bytearray(seqs[a][s0:s0 + ln])
            mut = rng.random(ln) < float(rng.choice([0.0, 0.03, 0.1]))
            sub = rng.integers(0, 4, size=ln)
            for i in mut.nonzero()[0]:
                seg[i] = b"ACGT"[sub[i]]
            if rng.random() < 0.5:
                seg = bytearray(bytes(seg).translate(comp)[::-1])
            seqs[b][t0:t0 + ln] = seg
        g = g[:-3] + f".par{int(rng.integers(1 << 30))}.fa"
        with open(g, "w") as f:
            for r, sq in zip(recs, seqs):
                f.write(">" + r[0] + "\n" + sq.decode() + "\n")
    # awkward query records: unmappable, very short, X / * / lower case, an empty one, a duplicate
    recs = open(p).read().split(">")[1:]
    aa = synth.AA20
    extra = [f"rnd{k}\n" + "".join(aa[i] for i in rng.integers(0, 20, size=int(rng.integers(1, 400)))) + "\n" for k in range(3)]
    extra.append("tiny\nMK\n")
    extra.append("empty\n\n")
    if recs:
        n0, s0 = recs[0].split("\n", 1)
        s0 = s0.replace("\n", "")
        extra.append("dup_" + n0 + "\n" + s0 + "\n")
        extra.append("lower_" + n0 + "\n" + s0.lower() + "\n")
        k = len(s0) // 2
        extra.append("xstar_" + n0 + "\n" + s0[:k] + "X*X" + s0[k + 3:] + "\n")
        extra.append("wrapped_" + n0 + " some comment\n" + "\n".join(s0[i:i + 60] for i in range(0, len(s0), 60)) + "\n")
    order = rng.permutation(len(recs) + len(extra))
    allrec = recs + extra
    p2 = p[:-4] + ".fuzz.faa"
    with open(p2, "w") as f:
        for i in order:
            f.write(">" + allrec[i])
    return g, p2


def random_options(rng, g, d):
    o = ["-t", str(int(rng.choice([1, 3])))]

    def maybe(p, *args):
        if rng.random() < p:
            o.extend(str(a) for a in args)

    if rng.random() < 0.15:
        o.append("-S")
    maybe(0.15, "-c", int(rng.choice([2, 50, 20000])))
    if rng.random() < 0.3:
        maybe(1.0, "-G", rng.choice(["500", "5k", "50k", "300k"]))
    elif rng.random() < 0.2:
        o.append("-I")
    maybe(0.15, "-w", rng.choice(["0", "0.3", "2"]))
    maybe(0.15, "-n", int(rng.integers(1, 6)))
    maybe(0.15, "-m", int(rng.choice([0, 20, 60])))
    maybe(0.15, "-l", int(rng.choice([4, 5, 6])))
    maybe(0.25, "-e", rng.choice(["100", "2k", "10k", "50k"]))
    maybe(0.2, "-p", rng.choice(["0", "0.3", "0.9", "1"]))
    maybe(0.2, "-N", int(rng.choice([0, 1, 5, 100])))
    maybe(0.3, "-O", int(rng.integers(1, 31)))
    maybe(0.3, "-E", int(rng.integers(0, 6)))
    maybe(0.3, "-J", int(rng.integers(3, 61)))
    maybe(0.15, "--J2", int(rng.integers(3, 61)))
    maybe(0.3, "-F", int(rng.integers(1, 61)))
    maybe(0.2, "-C", rng.choice(["0", "0.5", "1", "2.5"]))
    maybe(0.2, "-B", int(rng.integers(0, 21)))
    maybe(0.3, "-j", int(rng.integers(0, 3)))
    maybe(0.15, "--xdrop", int(rng.choice([5, 30, 400])))
    maybe(0.15, "--ie-coef", rng.choice(["0", "0.25", "1", "2.5"]))
    maybe(0.1, "--max-skip", int(rng.choice([0, 3, 100])))
    maybe(0.1, "--max-intron-out", int(rng.choice([0, 10, 1000])))
    maybe(0.1, "-g", int(rng.choice([10, 100, 5000])))
    if rng.random() < 0.1:
        o.append("--no-pre-chain")
    if rng.random() < 0.05:
        o.append("-A")
    if rng.random() < 0.3:
        o.append("-u")
    maybe(0.2, "--outn", int(rng.choice([1, 2, 1000])))
    maybe(0.2, "--outs", rng.choice(["0", "0.5", "0.99", "1"]))
    maybe(0.2, "--outc", rng.choice(["0", "0.5", "0.9"]))
    maybe(0.3, "-K", rng.choice(["1", "500", "3k", "1M"]))
    fmt = rng.random()
    if fmt < 0.15:
        o.append("--gff")
    elif fmt < 0.25:
        o.append("--gff-only")
    elif fmt < 0.35:
        o.append("--gtf")
    if rng.random() < 0.15:
        o.append("--aln")
    if rng.random() < 0.15:
        o.append("--trans")
    if rng.random() < 0.1:
        o.append("--no-cs")
    maybe(0.1, "-P", "ZZ")
    maybe(0.1, "--gff-delim", "#")
    if rng.random() < 0.2:
        sp = synth.make_spsc(g, os.path.join(d, f"s{int(rng.integers(1 << 30))}.spsc"), seed=int(rng.integers(1, 1000)))
        o.extend(["--spsc", sp])
        maybe(0.3, "--spsc0", int(rng.integers(0, 15)))
        maybe(0.3, "--spsc-max", int(rng.integers(0, 15)))
    if rng.random() < float(os.environ.get("MPB_FUZZ_P_INDEX", 0.08)):  # index options (host index builder; the default index is what the GPU stages are built for)
        maybe(0.5, "-M", int(rng.choice([0, 2])))
        maybe(0.5, "-L", int(rng.choice([10, 50])))
        maybe(0.3, "-b", int(rng.choice([7, 9])))
        maybe(0.3, "-k", 5)
        maybe(0.4, "-T", int(rng.choice([2, 3, 4, 5, 6, 9, 11, 12, 13, 14, 16, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31, 33])))
    return o


def fuzz(seed, n_it, workdir=None):
    cli = os.environ.get("MPB_FUZZ_CLI") or build_cli()  # MPB_FUZZ_CLI: e.g. the same program built with -fsanitize=address,undefined
    if cli is None or not os.path.exists(REF_BIN):
        print("needs oracle/_ref/miniprot and oracle/_ref/miniprot_hostcheck_cli (oracle/Makefile)")
        return 0, 0
    rng = np.random.default_rng(seed)
    bad = n_ref_abort = 0
    with tempfile.TemporaryDirectory(dir=workdir) as d:
        for it in range(n_it):
            if it and it % 100 == 0:
                print(f"progress seed {seed}: {it} command lines, {bad} mismatches ({n_ref_abort} skipped: the reference aborted)", flush=True)
                for f in os.listdir(d):  # inputs of earlier iterations
                    if f not in (os.path.basename(g), os.path.basename(p)) and not f.endswith(".planted.faa"):
                        os.remove(os.path.join(d, f))
            if it % 4 == 0:
                g, p = random_inputs(rng, d)
            opts = random_options(rng, g, d)
            use_mpi = rng.random() < 0.15  # through a dumped index (mp_idx_dump / mp_idx_restore of either side, crosswise)
            outs = []
            mpi = [os.path.join(d, f"i{k}.mpi") for k in range(2)]
            if use_mpi:
                idx_opts = [x for i, x in enumerate(opts) if x in ("-M", "-L", "-b", "-k", "-T") or (i and opts[i - 1] in ("-M", "-L", "-b", "-k", "-T"))]
                for k, binary in enumerate((REF_BIN, cli)):
                    subprocess.run([binary, "-t2", "-d", mpi[k]] + idx_opts + [g], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            for k, binary in enumerate((REF_BIN, cli)):
                r = subprocess.run([binary] + opts + [mpi[1 - k] if use_mpi else g, p], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
                outs.append((r.returncode, r.stdout, r.stderr))
            if outs[0][0] < 0:  # the reference itself stopped at one of its assertions (e.g. align.c:200 with a tiny -J): nothing to compare with
                n_ref_abort += 1
                continue
            same = outs[0][0] == outs[1][0] and outs[0][1] == outs[1][1]
            same = same and b"Sanitizer" not in outs[1][2] and b"runtime error" not in outs[1][2]
            if use_mpi:
                same = same and open(os.path.join(d, "i0.mpi"), "rb").read() == open(os.path.join(d, "i1.mpi"), "rb").read()
            if not same:
                bad += 1
                keep = os.path.join(workdir or tempfile.gettempdir(), f"fuzz_cli_fail_s{seed}_i{it}")
                os.makedirs(keep, exist_ok=True)
                subprocess.run(["cp", g, p, keep])
                for k, nm in enumerate(("ref", "ours")):
                    open(os.path.join(keep, nm + ".out"), "wb").write(outs[k][1])
                    open(os.path.join(keep, nm + ".err"), "wb").write(outs[k][2])
                print(f"MISMATCH seed={seed} it={it} rc={outs[0][0]}/{outs[1][0]} opts={' '.join(opts)} mpi={use_mpi} -> {keep}", flush=True)
    print(f"seed {seed}: {n_it} command lines, {bad} mismatches ({n_ref_abort} skipped: the reference aborted)")
    return n_it, bad


if __name__ == "__main__":
    sys.exit(1 if fuzz(int(sys.argv[1]) if len(sys.argv) > 1 else 1, int(sys.argv[2]) if len(sys.argv) > 2 else 50, sys.argv[3] if len(sys.argv) > 3 else None)[1] else 0)
