"""Parity of a whole configuration: ours (mpb_map_file on the GPU) against the reference CLI (oracle/_ref/miniprot) on the
same synthetic inputs, byte for byte.  Test / measurement infrastructure: the reference binary is only the checker.

  python tools/parity.py CONFIG [--opt "-I"] [--opt "-G 50k -e 2k"] ... [--dir DIR] [--json OUT]

Every --opt string is one run of both sides with those reference CLI options (a subset is understood on our side:
-I, -G, -e, -j, -S).  Prints one line per run with the md5s and the wall times; exit status 1 on any mismatch.  Where the
reference is not built, its output digests recorded in tests/golden stand in for it (tests/oracle_lib.py ref_cli; no times then)."""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import miniprot_b200 as mp  # noqa: E402
import oracle_lib as ol  # noqa: E402
from miniprot_b200 import synth  # noqa: E402


def parse_num(s: str) -> int:
    s = s.strip()
    mul = {"k": 1000, "K": 1000, "m": 1000000, "M": 1000000, "g": 1000000000, "G": 1000000000}
    if s[-1] in mul:
        return int(float(s[:-1]) * mul[s[-1]] + .499)
    return int(s)


def our_options(mi, optstr: str):
    """mp_mapopt_t for a reference option string (main.c:93-153 for the handful of options the parity runs use)."""
    mo = mp.mapopt()
    tok = optstr.split()
    i = 0
    while i < len(tok):
        t = tok[i]
        if t == "-I":
            mp.lib().mp_mapopt_set_max_intron(mo, mi.contents.nt.contents.l_seq)
        elif t == "-G":
            i += 1
            mo.max_intron = mo.bw = parse_num(tok[i])
        elif t == "-e":
            i += 1
            mo.max_ext = parse_num(tok[i])
        elif t == "-j":
            i += 1
            mo.sp_model = int(tok[i])
        elif t == "-S":
            mo.flag |= mp.MP_F_NO_SPLICE  # main.c:130
            mo.bw = mo.max_intron = mo.max_ext = 1000
            mo.io = mo.io_end = 10000
        else:
            raise SystemExit(f"option {t} is not understood by tools/parity.py")
        i += 1
    return mo


def run_config(cfg: str, opts, d: str, threads: int, ctx=None, keep=False):
    spec = synth.CONFIGS[cfg]
    t0 = time.time()
    g, p = synth.generate(spec, d)
    t_gen = time.time() - t0
    mpi = os.path.join(d, spec.tag() + ".mpi")
    t0 = time.time()
    if not os.path.exists(mpi):
        mi0 = mp.idx_load(g, threads)
        mp.lib().mp_idx_dump((mpi + ".tmp").encode(), mi0)
        os.replace(mpi + ".tmp", mpi)
        mp.lib().mp_idx_destroy(mi0)
    t_build = time.time() - t0
    t0 = time.time()
    mi = mp.idx_load(mpi)
    t_load = time.time() - t0
    own = ctx is None
    if own:
        ctx = mp.Context(0)
    t0 = time.time()
    assert mp.lib().mpb_idx_upload(ctx.h, mi) == 0
    t_up = time.time() - t0
    n_prot = sum(1 for line in open(p) if line.startswith(">"))
    rows = []
    for o in opts:
        mo = our_options(mi, o)
        out = os.path.join(d, "ours.paf")
        ctx.reset_stats()
        t0 = time.time()
        mp.map_file(ctx, mi, p, out, mo)
        t_ours = time.time() - t0
        st = ctx.stats()
        want = ol.ref_cli(o.split(), g, p, threads=threads, index=mpi)  # the reference restores the same index file
        t_ref = want.get("s")
        t_ref_map = None
        for line in want.get("err", b"").decode().splitlines():  # "[M::mp_idx_restore@0.210*1.00] ..." (index.c:227): mapping = wall - restore
            if "mp_idx_restore@" in line:
                try:
                    t_ref_map = t_ref - float(line.split("mp_idx_restore@")[1].split("*")[0])
                except Exception:
                    pass
        ours = open(out, "rb").read()
        same = hashlib.md5(ours).hexdigest() == want["md5"]
        row = {"config": cfg, "opt": o, "identical": same, "n_proteins": n_prot, "paf_lines": ours.count(b"\n"), "ref_lines": want["lines"],
               "md5_ours": hashlib.md5(ours).hexdigest(), "md5_ref": want["md5"], "ours_s": round(t_ours, 3), "ref_s": None if t_ref is None else round(t_ref, 3),
               "ref_map_s": None if t_ref_map is None else round(t_ref_map, 3), "ref_threads": threads if t_ref is not None else None,
               "anchors_per_protein": st.n_anchors / max(n_prot, 1), "dp_gcells": (st.dp_cells_ext + st.dp_cells_tb) / 1e9,
               "wall_ms": [round(x, 1) for x in st.ms_wall], "gen_s": round(t_gen, 1), "idx_build_s": round(t_build, 1), "idx_load_s": round(t_load, 2),
               "idx_upload_s": round(t_up, 2)}
        if not same and "out" in want:
            a, b = ours.decode().splitlines(), want["out"].decode().splitlines()
            row["first_diffs"] = [(x[:160], y[:160]) for x, y in zip(a, b) if x != y][:3]
            if keep:
                open(os.path.join(d, "ref.paf"), "wb").write(want["out"])
        rows.append(row)
        print(json.dumps(row), flush=True)
    mp.lib().mp_idx_destroy(mi)
    if own:
        ctx.close()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("config")
    ap.add_argument("--opt", action="append", default=[])
    ap.add_argument("--dir", default=os.environ.get("MPB_BENCH_DIR", "/tmp/mpb_bench"))
    ap.add_argument("--json", default=None)
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 8)
    ap.add_argument("--keep", action="store_true")
    a = ap.parse_args()
    rows = run_config(a.config, a.opt or [""], os.path.join(a.dir, a.config), a.threads, keep=a.keep)
    if a.json:
        with open(a.json, "w") as f:
            json.dump(rows, f, indent=1)
    sys.exit(0 if all(r["identical"] for r in rows) else 1)


if __name__ == "__main__":
    main()
