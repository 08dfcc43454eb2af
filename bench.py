#!/usr/bin/env python
"""bench.py -- the protein-to-genome mapping hot path on N B200s (BASELINE.json metric: proteins/s, DP Gcell/s).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload C2|C5|C4s|C3s|small|tiny]
                  [--dump-outputs DIR]

One "step" = one pass of the hot path (seed + chain + refine + nasw DP waves + host bookkeeping) over one batch of
synthetic proteins of the named workload (C2 = BASELINE.json configs[1]: 100 Mbp genome, 1000 proteins of ~400 aa per GPU).
N>1 is launched by torchrun, one rank per GPU: rank 0 loads the index, ONE NCCL broadcast puts ki / kb / packed genome
into every GPU's HBM, every rank then maps its own shard of queries (weak scaling) with no further communication.

Both arms time MAPPING with the index already loaded (ours: resident in HBM; reference: resident in host memory), on the same
proteins: the N shards of 1000 proteins each.

  ours       `value`  = mpb_map_batch: parsed proteins in host memory -> regions (index resident in HBM)
             `e2e`    = mpb_map_file: FASTA file in -> PAF file out, every host<->device copy inside the timed region
  reference  `value` = `e2e` = the unmodified reference's own mp_map_file (oracle/_ref/libref.so, compiled from /root/reference by
             oracle/Makefile, all host threads) on the concatenation of the same N shards, FASTA in -> PAF out, called in-process
             with its index loaded once before the timed region.

What a process pays once (context creation, index load, upload / broadcast) is reported separately under `process`.
The PAF of EVERY rank is compared with the reference's output for that rank's shard, where the reference is built; a mismatch
fails the run.

--dump-outputs DIR writes what the last timed `value` step returned to its caller (rank 0's regions: coordinates, scores,
alignment statistics, CIGARs, exon features) as DIR/<name>.npy in float64, so that two builds can be compared output for output
on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from miniprot_b200 import synth  # noqa: E402

REF_BIN = os.path.join(ROOT, "oracle", "_ref", "miniprot")
REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libref.so")
CACHE = os.environ.get("MPB_BENCH_DIR", "/tmp/mpb_bench")
PHASES = ["S1_seed_chain", "H1_regions", "S2_refine", "H2_plan", "S3_dp_waves", "H3_finish"]
WORKLOAD_OPTS = {"C3": "-I", "C3s": "-I"}  # reference CLI options that belong to a workload (BASELINE.json configs[2])


def read_fasta(path):
    names, seqs = [], []
    with open(path) as f:
        for line in f:
            if line.startswith(">"):
                names.append(line[1:].split()[0])
                seqs.append([])
            else:
                seqs[-1].append(line.strip())
    return names, ["".join(s) for s in seqs]


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu=0):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag = gpu, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower().startswith("active") for r in self.rows if len(r) > 3 + k)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def prepare(workload, rank, world):
    """Synthetic inputs (rank 0 writes genome, planted proteins and every rank's query shard; the others wait outside)."""
    spec = synth.CONFIGS[workload]
    d = os.path.join(CACHE, workload)
    if rank == 0:
        synth.generate(spec, d)
        for r in range(world):
            synth.shard_queries(spec, d, r)
    return spec, d


class Extra(C.Structure):  # mp_extra_t (include/miniprot_b200.h), followed by n_cigar uint32 CIGAR words
    _fields_ = [(f, C.c_int32) for f in ("dp_score", "dp_max", "dp_max2", "n_cigar", "m_cigar", "blen", "n_fs", "n_stop", "dist_stop",
                                         "dist_start", "n_iden", "n_plus")]


class Feat(C.Structure):  # mp_feat_t
    _fields_ = [("vs", C.c_int64), ("ve", C.c_int64), ("qs", C.c_int32), ("qe", C.c_int32), ("type", C.c_int16), ("phase", C.c_int16),
                ("n_fs", C.c_int32), ("n_stop", C.c_int32), ("score", C.c_int32), ("n_iden", C.c_int32), ("blen", C.c_int32),
                ("donor", C.c_char * 2), ("acceptor", C.c_char * 2)]


class Reg1(C.Structure):  # mp_reg1_t
    _fields_ = [(f, C.c_int32) for f in ("off", "cnt", "id", "parent", "n_sub", "subsc", "n_feat", "m_feat", "n_exon", "chn_sc", "chn_sc_ungap")] + \
        [("hash", C.c_uint32), ("vid", C.c_uint32), ("qs", C.c_int32), ("qe", C.c_int32), ("vs", C.c_int64), ("ve", C.c_int64),
         ("a", C.c_void_p), ("feat", C.POINTER(Feat)), ("p", C.POINTER(Extra))]


REG_FIELDS = ("vid", "qs", "qe", "vs", "ve", "id", "parent", "n_sub", "subsc", "cnt", "n_exon", "n_feat", "chn_sc", "chn_sc_ungap", "hash")
EXTRA_FIELDS = ("dp_score", "dp_max", "dp_max2", "n_cigar", "blen", "n_fs", "n_stop", "dist_stop", "dist_start", "n_iden", "n_plus")
FEAT_FIELDS = ("vs", "ve", "qs", "qe", "type", "phase", "n_fs", "n_stop", "score", "n_iden", "blen")
DUMP_LIMIT = 64 << 20


def dump_regions(out_dir, n, n_reg, regs):
    """Every region of every protein (reg_*: one row per region, protein by protein; reg_qid = the protein's index in the batch,
    reg_has_extra = 0 where the region carries no alignment), the alignment statistics (ext_*), the CIGAR words of all regions
    concatenated (cigar, with reg_cigar_off), and the exon features (feat_*, with reg_feat_off).  All float64 (exact for these
    integers).  Above 64 MB in all, a fixed seeded sample of the proteins is written instead."""
    import numpy as np

    def arrays(qids):
        cols = {k: [] for k in ("reg_qid", "reg_has_extra", "reg_cigar_off", "reg_feat_off", "cigar")}
        cols.update({"reg_" + f: [] for f in REG_FIELDS})
        cols.update({"ext_" + f: [] for f in EXTRA_FIELDS})
        cols.update({"feat_" + f: [] for f in FEAT_FIELDS})
        for i in qids:
            rs = C.cast(regs[i], C.POINTER(Reg1))
            for j in range(n_reg[i]):
                r = rs[j]
                cols["reg_qid"].append(i)
                for f in REG_FIELDS:
                    cols["reg_" + f].append(getattr(r, f))
                cols["reg_cigar_off"].append(len(cols["cigar"]))
                cols["reg_feat_off"].append(len(cols["feat_vs"]))
                cols["reg_has_extra"].append(1 if r.p else 0)
                e = r.p.contents if r.p else Extra()
                for f in EXTRA_FIELDS:
                    cols["ext_" + f].append(getattr(e, f))
                if r.p and e.n_cigar:
                    cig = C.cast(C.addressof(e) + C.sizeof(Extra), C.POINTER(C.c_uint32 * e.n_cigar)).contents
                    cols["cigar"].extend(cig)
                for k in range(r.n_feat if r.feat else 0):
                    for f in FEAT_FIELDS:
                        cols["feat_" + f].append(getattr(r.feat[k], f))
        return {k: np.asarray(v, dtype=np.float64) for k, v in cols.items()}

    out = arrays(range(n))
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT:
        keep = np.sort(np.random.default_rng(0).permutation(n)[:max(1, int(n * DUMP_LIMIT / total * 0.9))])
        out = arrays(keep)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def workload_text(name, spec, n_per_gpu, world):
    return (f"{name}: {spec.genome_len} bp genome, {world} x {n_per_gpu} proteins ~400 aa (one shard per GPU), identity {spec.identity}, "
            f"options '{WORKLOAD_OPTS.get(name, '')}'")


# ---------------------------------------------------------------------------------------------------------------------------
# the reference, in-process (oracle/_ref/libref.so: every symbol of the unmodified reference renamed ref_*)
class RefLib:
    def __init__(self):
        import miniprot_b200 as mp  # only for the ctypes mirrors of the option structs (same layout: miniprot.h:36-77)

        self.mp = mp
        self.L = C.CDLL(REF_LIB)
        self.L.ref_mp_start()
        C.c_int32.in_dll(self.L, "ref_mp_verbose").value = 1
        self.L.ref_mp_idx_load.restype = C.c_void_p
        self.L.ref_mp_idx_load.argtypes = [C.c_char_p, C.c_void_p, C.c_int32]
        self.L.ref_mp_map_file.restype = C.c_int32
        self.L.ref_mp_map_file.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int]
        self.L.ref_mp_idx_destroy.argtypes = [C.c_void_p]
        self.L.ref_mp_mapopt_set_max_intron.argtypes = [C.c_void_p, C.c_int64]
        self.libc = C.CDLL(None)
        self.mi = None

    def load(self, path, threads):
        io = self.mp.IdxOpt()
        self.L.ref_mp_idxopt_init(C.byref(io))
        t0 = time.perf_counter()
        self.mi = self.L.ref_mp_idx_load(path.encode(), C.byref(io), threads)
        if not self.mi:
            raise RuntimeError(f"reference cannot load {path}")
        return time.perf_counter() - t0

    def mapopt(self, workload, l_seq):
        mo = self.mp.MapOpt()
        self.L.ref_mp_mapopt_init(C.byref(mo))
        if WORKLOAD_OPTS.get(workload) == "-I":
            self.L.ref_mp_mapopt_set_max_intron(C.byref(mo), l_seq)
        return mo

    def map_file(self, prot, out_path, mo, threads):
        """ref mp_map_file writes to stdout: point fd 1 at out_path for the duration of the call.  Returns seconds."""
        sys.stdout.flush()
        self.libc.fflush(None)
        saved = os.dup(1)
        fd = os.open(out_path, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o644)
        os.dup2(fd, 1)
        os.close(fd)
        try:
            t0 = time.perf_counter()
            rc = self.L.ref_mp_map_file(self.mi, prot.encode(), C.byref(mo), threads)
            self.libc.fflush(None)
            dt = time.perf_counter() - t0
        finally:
            os.dup2(saved, 1)
            os.close(saved)
        if rc != 0:
            raise RuntimeError("reference mp_map_file failed")
        return dt

    def close(self):
        if self.mi:
            self.L.ref_mp_idx_destroy(self.mi)
            self.mi = None


def ensure_ref_index(spec, d, cores):
    g = os.path.join(d, spec.tag() + ".fa")
    mpi = os.path.join(d, spec.tag() + ".ref.mpi")
    if not os.path.exists(mpi):
        subprocess.run([REF_BIN, f"-t{cores}", "-d", mpi + ".tmp", g], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        os.replace(mpi + ".tmp", mpi)
    return mpi


def run_reference(args):
    """--impl reference: the unmodified reference's mp_map_file on this box's host cores, same proteins, index preloaded."""
    world = max(args.gpus, 1)
    cores = os.cpu_count() or 1
    if not os.path.exists(REF_LIB):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libref.so is not built (run __graft_entry__.build() where /root/reference exists)"}))
        return
    spec, d = prepare(args.workload, 0, world)
    mpi = ensure_ref_index(spec, d, cores)
    shards = [synth.shard_queries(spec, d, r) for r in range(world)]
    allp = os.path.join(d, f"{spec.tag()}.all{world}.faa")
    with open(allp, "w") as o:
        for s in shards:
            o.write(open(s).read())
    n_prot = len(read_fasta(allp)[0])
    ref = RefLib()
    t_load = ref.load(mpi, cores)
    l_seq = os.path.getsize(os.path.join(d, spec.tag() + ".fa"))  # only used by -I workloads (set from the genome size, options.c:31)
    mo = ref.mapopt(args.workload, l_seq)
    out = os.path.join(d, "ref.all.paf")
    for _ in range(args.warmup):
        ref.map_file(allp, out, mo, cores)
    dts = [ref.map_file(allp, out, mo, cores) for _ in range(args.steps)]
    ref.close()
    dt = sum(dts) / len(dts)
    v = n_prot / dt
    print(json.dumps({
        "impl": "reference", "metric": "proteins/s", "value": v, "unit": "proteins/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16 (SSE2, 8 lanes)", "data": "synthetic",
        "config": {"workload": workload_text(args.workload, spec, n_prot // world, world), "timed": "mp_map_file in-process (FASTA in, PAF out), index resident in host memory"},
        "process": {"index_load_s": round(t_load, 3), "note": "mp_idx_load of the prebuilt .mpi, once, outside the timed region"},
        "cpu_baseline": {"value": v, "unit": "proteins/s", "cores": cores, "kind": "reference",
                         "sample": f"all {n_prot} proteins ({world} shards), mp_map_file with {cores} threads, {args.steps} timed passes of {dt:.2f} s"},
        "e2e": {"value": v, "unit": "proteins/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ---------------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write rank 0's results of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))

    if args.impl == "reference":
        if rank == 0:
            run_reference(args)
        return

    t_proc = time.perf_counter()
    import numpy as np
    import torch
    import miniprot_b200 as mp

    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    L = mp.lib()
    L.mpb_event_end_ms.restype = C.c_double
    L.mpb_event_begin.argtypes = [C.c_void_p]
    L.mpb_event_end_ms.argtypes = [C.c_void_p]
    L.mpb_map_batch.argtypes = [C.c_void_p, C.POINTER(mp.Idx), C.POINTER(mp.MapOpt), C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mpb_regs_free.argtypes = [C.c_int32, C.c_void_p, C.c_void_p]
    cores = os.cpu_count() or 1

    spec, d = prepare(args.workload, rank, world)
    g = os.path.join(d, spec.tag() + ".fa")
    mpi = os.path.join(d, spec.tag() + ".mpi")
    t_build = 0.0
    if rank == 0 and not os.path.exists(mpi):
        t0 = time.perf_counter()
        mi0 = mp.idx_load(g, cores)
        L.mp_idx_dump((mpi + ".tmp").encode(), mi0)
        os.replace(mpi + ".tmp", mpi)
        L.mp_idx_destroy(mi0)
        t_build = time.perf_counter() - t0
    if dist:
        dist.barrier()
    t0 = time.perf_counter()
    ctx = mp.Context(local)  # pins this rank's host threads to the GPU's NUMA node (MPB_AFFINITY=0 disables)
    t_ctx = time.perf_counter() - t0
    class DevMem:  # a device buffer of the library as a torch tensor (zero copy, __cuda_array_interface__)
        def __init__(self, ptr, n, typestr):
            self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3}

    bcast_ms = None
    t0 = time.perf_counter()
    if not dist:
        mi = mp.idx_load_device(ctx, mpi)  # .mpi -> HBM through pinned staging buffers; only the genome section stays on the host
        t_load, t_up = time.perf_counter() - t0, 0.0
    else:
        # rank 0 loads the file into its HBM; the ONE collective of the path -- an NCCL broadcast of ki / kb / packed genome over
        # NVLink -- fills the other GPUs, whose ranks read only the head of the file (contig table, genome for the host phases)
        mi = mp.idx_load_device(ctx, mpi) if rank == 0 else L.mpb_idx_load_meta(mpi.encode())
        assert mi
        t_load = time.perf_counter() - t0
        t0 = time.perf_counter()
        nb = mp.n_bucket(mi.contents.opt)
        n_kb, l_seq = mi.contents.n_kb, mi.contents.nt.contents.l_seq
        if rank == 0:
            pk, pb, ps = C.c_void_p(), C.c_void_p(), C.c_void_p()
            assert L.mpb_idx_device_ptrs(ctx.h, C.byref(pk), C.byref(pb), C.byref(ps)) == 0
            ki = torch.as_tensor(DevMem(pk.value, nb + 1, "<i8"), device=dev)
            kb = torch.as_tensor(DevMem(pb.value, max(n_kb, 1), "<i4"), device=dev)
            sq = torch.as_tensor(DevMem(ps.value, (l_seq + 1) // 2, "|u1"), device=dev)
        else:
            ki = torch.empty(nb + 1, dtype=torch.int64, device=dev)
            kb = torch.empty(max(n_kb, 1), dtype=torch.int32, device=dev)
            sq = torch.empty((l_seq + 1) // 2, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for t in (ki, kb, sq):
            dist.broadcast(t, 0)
        e1.record()
        torch.cuda.synchronize()
        bcast_ms = e0.elapsed_time(e1)
        if rank != 0:
            assert L.mpb_idx_attach_device(ctx.h, mi, ki.data_ptr(), kb.data_ptr(), sq.data_ptr()) == 0
        t_up = time.perf_counter() - t0
    l_seq = mi.contents.nt.contents.l_seq

    shard = int(os.environ.get("MPB_BENCH_SHARD", rank))  # (diagnostics: map another rank's shard on this GPU)
    if shard != rank:
        synth.shard_queries(spec, d, shard)
    prot = synth.shard_queries(spec, d, shard)
    names, seqs = read_fasta(prot)
    n = len(seqs)
    mo = mp.mapopt()
    if WORKLOAD_OPTS.get(args.workload) == "-I":
        L.mp_mapopt_set_max_intron(mo, l_seq)
    c_seqs = (C.c_char_p * n)(*[s.encode() for s in seqs])
    c_names = (C.c_char_p * n)(*[s.encode() for s in names])
    c_lens = (C.c_int32 * n)(*[len(s) for s in seqs])
    n_reg = (C.c_int32 * n)()
    regs = (C.c_void_p * n)()
    out_paf = os.path.join(d, f"ours.rank{rank}.paf")

    def step_resident(keep=False):
        """keep: leave the regions to the caller (the last timed step: dumped if asked, and freed, after the timed region)."""
        assert L.mpb_map_batch(ctx.h, mi, C.byref(mo), n, c_seqs, c_lens, c_names, n_reg, regs) == 0
        if not keep:
            L.mpb_regs_free(n, n_reg, regs)

    def step_e2e(keep=False):
        mp.map_file(ctx, mi, prot, out_paf, mo)

    def timed(fn, steps):
        """K steps between barriers + device synchronisation; CUDA events on the context's stream and the host clock around
        them (a step ends with host bookkeeping after the last kernel, so the larger of the two closes the bracket)."""
        if dist:
            dist.barrier()
        torch.cuda.synchronize()
        L.mpb_event_begin(ctx.h)
        t0 = time.perf_counter()
        for i in range(steps):
            fn(keep=i == steps - 1)
        ms = L.mpb_event_end_ms(ctx.h)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        mine = max(ms, wall)
        ms = mine
        if dist:
            t = torch.tensor([mine], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, mine

    t0 = time.perf_counter()
    step_e2e()  # first pass of this process: grows the arenas (cudaMalloc), loads the kernels
    t_first = time.perf_counter() - t0
    for _ in range(max(args.warmup, 3)):
        step_resident()
    ctx.reset_stats()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, ms_mine = timed(step_resident, args.steps)
    st = ctx.stats()
    if args.dump_outputs is not None and rank == 0:
        dump_regions(args.dump_outputs, n, n_reg, regs)
    L.mpb_regs_free(n, n_reg, regs)
    step_e2e()
    ctx.reset_stats()
    ms_e2e, ms_e2e_mine = timed(step_e2e, args.steps)
    st2 = ctx.stats()
    sampler.stop_flag = True
    int_peak = None
    if rank == 0:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import int_peak as ip
        int_peak = ip.measure(ctx)

    # ---- parity, EVERY rank: this rank's PAF against the reference's mp_map_file on the same shard (the checker only)
    parity, cpu = None, None
    if os.path.exists(REF_LIB) and os.path.exists(REF_BIN):
        if rank == 0:
            ensure_ref_index(spec, d, cores)
        if dist:
            dist.barrier()
        try:
            os.sched_setaffinity(0, range(cores))  # the context pinned this process to the GPU's NUMA node; the checker may use every core
        except Exception:
            pass
        ref = RefLib()
        thr = max(cores // world, 1)
        ref.load(os.path.join(d, spec.tag() + ".ref.mpi"), thr)
        ref_out = os.path.join(d, f"ref.rank{rank}.paf")
        ref_dt = ref.map_file(prot, ref_out, ref.mapopt(args.workload, l_seq), thr)
        ref.close()
        parity = open(out_paf, "rb").read() == open(ref_out, "rb").read()
        cpu = {"value": n / ref_dt, "unit": "proteins/s", "cores": thr, "kind": "reference",
               "sample": f"the {n} proteins of rank 0's shard, reference mp_map_file in-process with {thr} threads, index resident, {ref_dt:.2f} s"}
    per_rank = [[ms_mine / args.steps, ms_e2e_mine / args.steps, 1.0 if parity else 0.0 if parity is not None else -1.0] + [w / args.steps for w in st.ms_wall]]
    if dist:
        t = torch.tensor(per_rank[0], dtype=torch.float64, device=dev)
        allt = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank = [[float(x) for x in a.tolist()] for a in allt]

    tot_prot = n * world
    value = tot_prot / (ms / args.steps / 1e3)
    e2e = tot_prot / (ms_e2e / args.steps / 1e3)
    cells = (st.dp_cells_ext + st.dp_cells_tb) / args.steps
    if rank != 0:
        ctx.close()
        if dist:
            dist.destroy_process_group()
        return

    parity_all = None if any(r[2] < 0 for r in per_rank) else all(r[2] > 0.5 for r in per_rank)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)

    # ---- rooflines (DESIGN.md section 4).  Kernel times are CUDA events on the stream each class is launched on.
    CLS = ["v3<1>", "v3<2>", "v3<4>", "v3<8>", "cols<1>", "cols<2>", "cols<4>", "cols<8>", "cols<8,multi>", "pair<1>", "v3<4> x 2 column passes", "", "", "", "", ""]

    def cls_rows(b):
        rows = []
        for c in range(16):
            if st.n_class[b][c]:
                rows.append({"kernel": ("nasw_tb " if b else "nasw_ext ") + CLS[c], "launches_per_step": st.n_class[b][c] / args.steps,
                             "ms_per_launch": st.ms_class[b][c] / st.n_class[b][c], "gcell_per_launch": st.cells_class[b][c] / st.n_class[b][c] / 1e9})
        return rows
    ext_rows, tb_rows = cls_rows(0), cls_rows(1)
    # HBM roofline: the traceback kernels write 2 B per DP cell once (SURVEY 8d); the class with the most cells is quoted
    roofline = {"bound": "hbm", "kernel": None, "achieved": None, "peak": hbm_peak, "unit": "GB/s", "frac": None, "traffic": None}
    if tb_rows:
        top = max(tb_rows, key=lambda r: r["gcell_per_launch"] * r["launches_per_step"])
        gbs = top["gcell_per_launch"] * 2 / (top["ms_per_launch"] / 1e3)
        traffic = None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
            if args.workload == "C2":
                traffic = tr.get(top["kernel"], {}).get("dram_bytes_per_launch")
        except Exception:
            pass
        roofline.update({"kernel": top["kernel"] + " (global alignment with traceback; 2 B per DP cell written once)", "achieved": gbs, "frac": gbs / hbm_peak,
                         "traffic": traffic, "algorithmic_bytes_per_launch": top["gcell_per_launch"] * 2e9, "ms_per_launch": top["ms_per_launch"],
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6.65 TB/s (of fallback)"})
    # integer roofline of the dominant kernel by time (score-only extension): 32 int16 operations per cell (SURVEY 8d) against
    # the measured fused add-max rate of this device (tools/int_peak.py, run above)
    roofline_int = None
    if ext_rows and int_peak:
        top = max(ext_rows, key=lambda r: r["ms_per_launch"] * r["launches_per_step"])
        ach = top["gcell_per_launch"] * 32e9 / (top["ms_per_launch"] / 1e3)
        pk32, pk16 = int_peak["viaddmnmx_s32"]["int_ops_per_s"], int_peak["viaddmnmx_s16x2"]["int_ops_per_s"]
        roofline_int = {"bound": "int", "kernel": top["kernel"] + " (score-only extension)", "achieved": ach / 1e12, "peak": pk16 / 1e12, "unit": "Tint16-op/s",
                        "frac": ach / pk16, "peak_32bit_lanes": pk32 / 1e12, "frac_of_32bit_peak": ach / pk32, "ops_per_cell": 32, "ms_per_launch": top["ms_per_launch"],
                        "note": "peak = measured VIADDMNMX.S16x2 issue rate x 4 ops (tools/int_peak.py); the wave is bounded by the row-to-row latency of its longest problems"}
    walls = sorted(r[0] for r in per_rank)
    slow = max(range(world), key=lambda r: per_rank[r][0])
    print(json.dumps({
        "metric": "proteins/s", "value": value, "unit": "proteins/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16 scores",
        "data": "synthetic",
        "config": {"workload": workload_text(args.workload, spec, n, world), "timed": "mapping with the index resident in HBM (value: mpb_map_batch; e2e: mpb_map_file, FASTA in, PAF out)",
                   "l2": "index (ki+kb+genome, 315 MB at C2) and DP working set exceed the 126 MB L2; no flush needed",
                   "paf_identical_to_reference": parity_all, "paf_identical_per_rank": [r[2] > 0.5 for r in per_rank]},
        "process": {"ctx_create_s": round(t_ctx, 3), "index_load_s": round(t_load, 3), "index_broadcast_s": round(t_up, 3), "index_build_s": round(t_build, 2),
                    "nccl_index_broadcast_ms": bcast_ms, "first_pass_s": round(t_first, 3), "since_start_s": round(time.perf_counter() - t_proc, 1),
                    "note": "paid once per process, outside the timed region (the reference arm reports its own index_load_s)"},
        "dp_gcell_per_s": cells / (ms / args.steps / 1e3) / 1e9 * world,
        "stage_ms_per_step": {"seed": st.ms_seed / args.steps, "chain": st.ms_chain / args.steps, "refine": st.ms_refine / args.steps,
                              "dp_prep": st.ms_prep / args.steps, "dp_waves_wall": st.ms_dp_wave / args.steps, "dp_backtrack": st.ms_bt / args.steps},
        "nasw_kernels": ext_rows + tb_rows,
        "wall_ms_per_step": dict(zip(PHASES, [w / args.steps for w in st.ms_wall])),
        "ranks": {"ms_per_step": {"min": walls[0], "median": walls[len(walls) // 2], "max": walls[-1]}, "per_rank_ms_per_step": [round(r[0], 3) for r in per_rank],
                  "per_rank_e2e_ms_per_step": [round(r[1], 3) for r in per_rank], "slowest_rank": slow,
                  "slowest_rank_wall_ms_per_step": dict(zip(PHASES, [round(x, 3) for x in per_rank[slow][3:]]))},
        "e2e": {"value": e2e, "unit": "proteins/s", "h2d_bytes_per_step": st2.h2d_bytes // args.steps, "d2h_bytes_per_step": st2.d2h_bytes // args.steps,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(st.kernel_launches), "roofline": roofline, "roofline_int": roofline_int, "int_peak": int_peak, "cpu_baseline": cpu,
        "clocks": sampler.summary(), "build": mp.build_info()}))
    ctx.close()
    if dist:
        dist.destroy_process_group()
    if parity_all is False:
        sys.stderr.write("bench.py: PAF differs from the reference on at least one rank\n")
        sys.exit(1)


if __name__ == "__main__":
    main()
