#!/usr/bin/env python
"""bench.py -- aligned bases/sec of the seed-chain-extend hot path on B200, next to the unmodified reference on the host CPUs.

  python bench.py --gpus N --steps K --warmup W [--workload map-ont|map-hifi|splice|ava-ont]   # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K --warmup W [--workload ...]                 # the UNMODIFIED reference (oracle/_ref)

A "step" is one pass of the whole hot path (mm_sketch -> seeds -> chain -> ksw2 -> hits, i.e. mm_map semantics) over one batch of
synthetic reads. The default workload is BASELINE.json configs[1]: 100k x 10 kb ONT-profile reads vs a 3 Gbp uniform-random
reference in 24 contigs, `-x map-ont -c`; --workload selects configs[2..4] (map-hifi -a, splice -c, ava-ont). Data are synthetic
(device-side counter-based generators, minimap2_b200/csrc/synth.cu); the reference arm maps the same genome (written to FASTA)
and a bounded sample of the same reads.

JSON line (rank 0):
  value        whole-job aligned bases/s with the read bases already resident in HBM when the timed region starts
  e2e          the same metric through the C-ABI call mm_map_batch() with HOST buffers (H2D of the reads and D2H of all results
               inside the timed region)
  file_e2e     the same metric through mm_map_file() -- FASTA parsing, mapping, PAF/SAM formatting and writing, i.e. exactly what
               the reference arm's number contains (like for like with `--impl reference`)
  parity       the bounded sample mapped by BOTH arms through mm_map_file(): output lines compared one by one
  roofline     the dominant kernel (K3 ksw2) from CUDA events on the launch stream + per-stage figures
  cpu_baseline the reference's own CPU code (oracle/_ref/libminimap2_ref.so) on this box's host cores
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

MM_F_CIGAR, MM_F_OUT_SAM, MM_F_OUT_CG = 0x004, 0x008, 0x020

# BASELINE.json configs[1..4] (SURVEY 8d describes the synthetic inputs). err = (rate, substitution share, insertion share).
WORKLOADS = {
    "map-ont": dict(preset="map-ont", k=15, w=10, genome_mbp=3000.0, contigs=24, reads=100000, read_len=10000, err=(0.10, 0.40, 0.25),
                    kind="genomic", out="-c", metric="aligned bases/sec (map-ont, 10 kb reads)",
                    desc="%d synthetic %d bp ONT-profile reads (10%% err, sub/ins/del 40/25/35) vs synthetic %.0f Mbp reference (24 contigs), -x map-ont -c"),
    "map-hifi": dict(preset="map-hifi", k=19, w=19, genome_mbp=3000.0, contigs=24, reads=200000, read_len=15000, err=(0.005, 1 / 3., 1 / 3.),
                     kind="genomic", out="-a", metric="aligned bases/sec (map-hifi, 15 kb reads)",
                     desc="%d synthetic %d bp HiFi-profile reads (0.5%% err, sub/ins/del 1/1/1) vs synthetic %.0f Mbp reference (24 contigs), -x map-hifi -a"),
    "splice": dict(preset="splice", k=15, w=5, genome_mbp=3000.0, contigs=24, reads=500000, read_len=2000, err=(0.03, 1 / 3., 1 / 3.),
                   kind="cdna", out="-c", metric="aligned bases/sec (splice, 2 kb cDNA reads)",
                   desc="%d synthetic %d bp cDNA reads (exons 100-500 bp over GT..AG introns of 100 bp-50 kb, 3%% err) vs synthetic %.0f Mbp reference (24 contigs), -x splice -c"),
    "ava-ont": dict(preset="ava-ont", k=15, w=5, genome_mbp=50.0, contigs=1, reads=50000, read_len=20000, err=(0.10, 0.40, 0.25),
                    kind="ava", out="", metric="aligned bases/sec (ava-ont, 20 kb reads, all-vs-all)",
                    desc="all-vs-all overlap of %d synthetic %d bp ONT-profile reads (10%% err) drawn from a %.0f Mbp genome, -x ava-ont"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="map-ont", choices=sorted(WORKLOADS))
    # workload knobs (defaults = the BASELINE.json config); smaller values are for development only and are reported in config
    ap.add_argument("--genome-mbp", type=float, default=None)
    ap.add_argument("--reads", type=int, default=None)
    ap.add_argument("--read-len", type=int, default=None)
    ap.add_argument("--threads", type=int, default=0, help="host threads for orchestration / the reference arm (0 = all cores)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="reads in the bounded CPU sample (0 = sized from a calibration run)")
    ap.add_argument("--ref-budget-s", type=float, default=100.0, help="wall-clock target for all reference-arm steps together")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-file-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (per-read hit counts and rep_len, the hits of a fixed sample of reads) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs covers this repository's arm only (the reference arm's output is PAF/SAM text)")
    return a


# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md)"""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            rows = [l.strip().split(", ") for l in open(self.path) if l.strip()]
            sm = sorted(float(r[0]) for r in rows if r[0].replace(".", "").isdigit())
            if sm:
                out["sm_mhz"] = sm[len(sm) // 2]
                out["sm_max_mhz"] = max(float(r[1]) for r in rows)
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for k, nm in enumerate(names):
                if any(len(r) > 3 + k and r[3 + k].strip().lower() == "active" for r in rows):
                    out["reasons"].append(nm)
            os.unlink(self.path)
        except Exception:
            pass
        return out


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def physical_cores():
    try:
        seen = set()
        phys = core = None
        for line in open("/proc/cpuinfo"):
            if line.startswith("physical id"):
                phys = line.split(":")[1].strip()
            elif line.startswith("core id"):
                core = line.split(":")[1].strip()
            elif not line.strip():
                if phys is not None and core is not None:
                    seen.add((phys, core))
                phys = core = None
        return len(seen) or None
    except Exception:
        return None


class StdoutTo:
    """redirects the C-level stdout (fd 1) of this process to a file while a library writes its PAF/SAM records"""

    def __init__(self, path):
        self.path = path

    def __enter__(self):
        sys.stdout.flush()
        C.CDLL(None).fflush(None)
        self.saved = os.dup(1)
        fd = os.open(self.path, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o644)
        os.dup2(fd, 1)
        os.close(fd)
        return self

    def __exit__(self, *a):
        C.CDLL(None).fflush(None)
        os.dup2(self.saved, 1)
        os.close(self.saved)


def paf_aligned_bases(path, sam=False, all_records=False):
    """sum of query spans of the primary records (PAF: tp:A:P; SAM: neither secondary nor supplementary... the PAF rule is what the
    metric defines, SAM output is converted with the CIGAR's query span)"""
    bases = 0
    with open(path) as f:
        for line in f:
            if sam:
                if line.startswith("@"):
                    continue
                c = line.split("\t", 7)
                flag = int(c[1])
                if flag & 4 or flag & 0x100:
                    continue
                n, span = 0, 0
                for ch in c[5]:
                    if ch.isdigit():
                        n = n * 10 + ord(ch) - 48
                    else:
                        if ch in "MI=X":
                            span += n
                        n = 0
                bases += span
            elif all_records or "tp:A:P" in line or "tp:A:I" in line:
                c = line.split("\t", 5)
                bases += int(c[3]) - int(c[2])
    return bases


def apply_output_flags(mo, wl):
    if wl["out"] == "-c":
        mo.flag |= MM_F_CIGAR | MM_F_OUT_CG
    elif wl["out"] == "-a":
        mo.flag |= MM_F_CIGAR | MM_F_OUT_SAM
    else:
        mo.flag &= ~MM_F_CIGAR


# ---------------------------------------------------------------------------------------------------------------------
class Reference:
    """The UNMODIFIED reference (libminimap2_ref.so built from /root/reference by oracle/Makefile; loaded RTLD_LOCAL) through its own
    public API: mm_idx_reader_read (index build, untimed) and mm_map_file per step."""

    def __init__(self, wl, ref_fa, n_threads, log):
        from minimap2_b200 import api  # only the ctypes struct mirrors (IdxOpt/MapOpt share the reference's layout)
        from oracle_lib import REF_SO
        self.ok = os.path.exists(REF_SO)
        if not self.ok:
            return
        self.api, self.nthr = api, n_threads
        L = self.L = C.CDLL(REF_SO)
        L.mm_set_opt.argtypes = [C.c_char_p, C.POINTER(api.IdxOpt), C.POINTER(api.MapOpt)]
        L.mm_idx_reader_open.restype = C.c_void_p
        L.mm_idx_reader_open.argtypes = [C.c_char_p, C.POINTER(api.IdxOpt), C.c_char_p]
        L.mm_idx_reader_read.restype = C.c_void_p
        L.mm_idx_reader_read.argtypes = [C.c_void_p, C.c_int]
        L.mm_idx_reader_close.argtypes = [C.c_void_p]
        L.mm_mapopt_update.argtypes = [C.POINTER(api.MapOpt), C.c_void_p]
        L.mm_map_file.restype = C.c_int
        L.mm_map_file.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(api.MapOpt), C.c_int]
        L.mm_idx_destroy.argtypes = [C.c_void_p]
        C.c_int.in_dll(L, "mm_verbose").value = 1
        self.io, self.mo = api.IdxOpt(), api.MapOpt()
        L.mm_set_opt(None, C.byref(self.io), C.byref(self.mo))
        L.mm_set_opt(wl["preset"].encode(), C.byref(self.io), C.byref(self.mo))
        apply_output_flags(self.mo, wl)
        t0 = time.time()
        rdr = L.mm_idx_reader_open(ref_fa.encode(), C.byref(self.io), None)
        self.mi = L.mm_idx_reader_read(rdr, n_threads)
        L.mm_idx_reader_close(rdr)
        L.mm_mapopt_update(C.byref(self.mo), self.mi)
        self.t_idx = time.time() - t0
        log("reference index built in %.1fs on %d threads (mid_occ=%d)" % (self.t_idx, n_threads, self.mo.mid_occ))

    def map_file(self, reads_fa, out_path, mini_batch=None, n_threads=None):
        mo = self.api.MapOpt.from_buffer_copy(self.mo)
        if mini_batch:
            mo.mini_batch_size = int(mini_batch)
        with StdoutTo(out_path):
            t = time.time()
            self.L.mm_map_file(self.mi, reads_fa.encode(), C.byref(mo), n_threads or self.nthr)
            C.CDLL(None).fflush(None)
            dt = time.time() - t
        return dt

    def close(self):
        if self.ok and self.mi:
            self.L.mm_idx_destroy(self.mi)
            self.mi = None


def write_reads_fasta(path, buf, read_len, lo, hi):
    with open(path, "wb") as f:
        for i in range(lo, hi):
            f.write(b">r%d\n" % i)
            f.write(buf[i * read_len:(i + 1) * read_len].tobytes())
            f.write(b"\n")


def gen_reads(L, idx, wl, n, read_len, seed, buf):
    if wl["kind"] == "cdna":
        L.mmb_synth_cdna_reads(idx, n, read_len, seed, wl["err"][0], buf.ctypes.data)
    else:
        L.mmb_synth_reads(idx, n, read_len, seed, wl["err"][0], wl["err"][1], wl["err"][2], buf.ctypes.data)


DUMP_READS, DUMP_CIGAR_READS, DUMP_MAX_BYTES = 2048, 256, 64 << 20


def collect_outputs(api, n_regs, regs, rep_len):
    """What mm_map_batch() handed back, as float64 arrays: n_regs and rep_len of every read; for a fixed seeded sample of reads, every
    field of their mm_reg1_t hits and of the mm_extra_t behind them, and the CIGAR words of the hits of the first DUMP_CIGAR_READS
    sampled reads (hit h's words are cigar[hits.cigar_off[h]:][:hits.n_cigar[h]]; cigar_off is -1 for the other hits)"""
    n = len(n_regs)
    sample = np.sort(np.random.default_rng(0).permutation(n)[:DUMP_READS])
    reg_fields = [f for f, _ in api.Reg1._fields_ if f != "p"]
    ext_fields = [f for f, _ in api.Extra._fields_ if f != "capacity"]
    cols = {f: [] for f in ["read"] + reg_fields + ext_fields + ["cigar_off"]}
    cigar, n_words = [], 0
    for k, i in enumerate(sample):
        arr = C.cast(C.c_void_p(int(regs[i])), C.POINTER(api.Reg1)) if regs[i] else None
        for j in range(int(n_regs[i])):
            r = arr[j]
            cols["read"].append(i)
            for f in reg_fields:
                cols[f].append(getattr(r, f))
            ex = r.p.contents if r.p else None
            for f in ext_fields:
                cols[f].append(getattr(ex, f) if ex else 0)
            cols["cigar_off"].append(n_words if ex and k < DUMP_CIGAR_READS else -1)
            if ex and k < DUMP_CIGAR_READS:
                cigar.append(np.ctypeslib.as_array((C.c_uint32 * ex.n_cigar).from_address(C.addressof(ex) + C.sizeof(api.Extra))).copy())
                n_words += ex.n_cigar
    out = {"n_regs": np.asarray(n_regs, dtype=np.float64), "rep_len": np.asarray(rep_len, dtype=np.float64), "sample_reads": sample.astype(np.float64),
           "cigar": np.concatenate(cigar).astype(np.float64) if cigar else np.zeros(0)}
    out.update({"hits." + ("as" if f == "as_" else f): np.asarray(v, dtype=np.float64) for f, v in cols.items()})
    assert sum(a.nbytes for a in out.values()) <= DUMP_MAX_BYTES, "output dump above %d bytes" % DUMP_MAX_BYTES
    return out


def compare_outputs(a_path, b_path, log, sam=False):
    def lines(p):
        with open(p) as f:
            return [l.rstrip("\n") for l in f if not (sam and l.startswith("@"))]
    a, b = lines(a_path), lines(b_path)
    mism = abs(len(a) - len(b))
    shown = 0
    for x, y in zip(a, b):
        if x != y:
            mism += 1
            if shown < 3:
                log("parity mismatch:\n  ref: %s\n  got: %s" % (x[:300], y[:300]))
                shown += 1
    return len(a), len(b), mism


# ---------------------------------------------------------------------------------------------------------------------
def main():
    a = parse_args()
    wl = dict(WORKLOADS[a.workload])
    for key, val in (("genome_mbp", a.genome_mbp), ("reads", a.reads), ("read_len", a.read_len)):
        if val is not None:
            wl[key] = val
    n_reads, read_len, genome_mbp = int(wl["reads"]), int(wl["read_len"]), float(wl["genome_mbp"])
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    n_threads_all = os.cpu_count() or 1
    nthr = a.threads or max(1, n_threads_all // max(1, world))
    sam = wl["out"] == "-a"
    ava = wl["kind"] == "ava"  # all-vs-all overlap: no hit is marked primary (tp:A:S everywhere), every record counts
    # identical in both arms (the driver compares it); everything arm-specific lives in cpu_baseline / e2e / host
    cfg = {"workload": a.workload + ": " + wl["desc"] % (n_reads, read_len, genome_mbp), "preset": wl["preset"], "k": wl["k"], "w": wl["w"],
           "reads_per_step_per_gpu": n_reads, "read_len": read_len, "genome_mbp": genome_mbp,
           "l2_policy": "inputs larger than L2 (>=1 GB of read bases + multi-GB index touched every step)"}

    def log(msg):
        if rank == 0:
            print("[bench] " + msg, file=sys.stderr, flush=True)

    os.environ["MM_B200_DEVICE"] = str(local_rank)
    import torch
    dist_on = world > 1
    if a.impl == "reference" and rank != 0:
        return 0
    if dist_on and a.impl != "reference":
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    # host worker pool per rank: half of the logical CPUs for one rank (the scheduler's group threads must never wait for a core), three
    # quarters of the rank's share when several ranks divide the box (the host work per rank does not shrink with the rank count)
    os.environ.setdefault("MM_B200_HOST_THREADS", str(n_threads_all // 2 if world <= 1 else max(8, (3 * n_threads_all) // (4 * world))))
    import minimap2_b200 as mb  # noqa: F401
    from minimap2_b200 import api
    L = api._setup()
    L.mmb_synth_cdna_reads.restype = C.c_int
    L.mmb_synth_cdna_reads.argtypes = [C.POINTER(api.Idx), C.c_int, C.c_int, C.c_uint64, C.c_float, C.c_void_p]
    L.mmb_aligned_bases.restype = C.c_int64
    L.mmb_aligned_bases.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    L.mm_map_file.restype = C.c_int
    L.mm_map_file.argtypes = [C.POINTER(api.Idx), C.c_char_p, C.POINTER(api.MapOpt), C.c_int]
    tmp = tempfile.mkdtemp(prefix="mm2bench_")
    ref_fa, sample_fa, full_fa = os.path.join(tmp, "ref.fa"), os.path.join(tmp, "sample.fa"), os.path.join(tmp, "reads.fa")

    # ---------------- data + index (untimed) ----------------
    t0 = time.time()
    # Every rank builds the same index deterministically on its own GPU from the seed (the device build takes seconds).
    # A loaded (non-synthetic) index is broadcast instead: see minimap2_b200/dist.py (NCCL broadcast of the device arrays).
    # One rank builds (or, for a real genome, loads) the index; the others receive its device arrays by ONE NCCL broadcast over
    # NVLink/NVSwitch (minimap2_b200/dist.py) and are independent from then on: no collective on the per-read path (SURVEY 8e).
    bcast = None
    keep_idx_bufs = None
    if dist_on and a.impl != "reference" and wl["kind"] != "ava":
        from minimap2_b200 import dist as mdist
        gidx = L.mmb_synth_index(int(genome_mbp * 1e6), int(wl["contigs"]), 11, wl["w"], wl["k"], 14) if rank == 0 else None
        torch.cuda.synchronize(); dist.barrier()
        tb = time.perf_counter()
        gidx, keep_idx_bufs = mdist.broadcast_index(gidx, rank, src=0)
        torch.cuda.synchronize(); dist.barrier()
        tb = time.perf_counter() - tb
        nbytes = int(sum(int(t.numel()) for t in keep_idx_bufs))
        bcast = {"bytes": nbytes, "ms": 1e3 * tb, "gb_per_s": nbytes / 1e9 / tb, "ranks": world,
                 "what": "device index arrays (hash table, positions, 4-bit sequence, offsets, occurrence counts) from rank 0 to all ranks, one NCCL broadcast per array; wall time between barriers"}
        log("index broadcast: %.2f GB in %.0f ms (%.0f GB/s)" % (nbytes / 1e9, 1e3 * tb, nbytes / 1e9 / tb))
    else:
        gidx = L.mmb_synth_index(int(genome_mbp * 1e6), int(wl["contigs"]), 11, wl["w"], wl["k"], 14)
    buf = np.zeros(n_reads * read_len, dtype=np.uint8)
    gen_reads(L, gidx, wl, n_reads, read_len, 12 + 1000 * (rank if a.impl != "reference" else 0), buf)
    names = ["r%d" % i for i in range(n_reads)]
    if wl["kind"] == "ava":  # the index IS the read set
        write_reads_fasta(full_fa, buf, read_len, 0, n_reads)
        L.mm_idx_destroy(gidx)
        gidx = None
        ref_fa = full_fa
    log("synthetic genome + reads ready in %.1fs" % (time.time() - t0))

    def make_aligner():
        if wl["kind"] == "ava":
            al_ = api.Aligner(fn_idx_in=full_fa, preset=wl["preset"], n_threads=nthr)
        else:
            al_ = api.Aligner(preset=wl["preset"], _idx=gidx, n_threads=nthr)
        al_.map_opt.flag &= ~MM_F_CIGAR  # the Aligner class follows mappy (CIGAR on); the bench follows the CLI flags of the config
        apply_output_flags(al_.map_opt, wl)
        return al_

    # =====================================================================================================================
    if a.impl == "reference":
        if gidx is not None:
            L.mmb_idx_write_fasta(gidx, ref_fa.encode())
            L.mm_idx_destroy(gidx)
        R = Reference(wl, ref_fa, n_threads_all, log)
        if not R.ok:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libminimap2_ref.so missing"}))
            return 0
        # size the per-step sample from a calibration run so that all steps together take about --ref-budget-s
        ns = a.cpu_sample
        if ns <= 0:
            nc = min(n_reads, max(256, int(3e7 // read_len)))
            write_reads_fasta(sample_fa, buf, read_len, 0, nc)
            dt = R.map_file(sample_fa, sample_fa + ".paf")
            rate = nc / max(dt, 1e-3)
            ns = int(min(n_reads, max(nc, rate * a.ref_budget_s / max(1, a.steps + a.warmup))))
            log("calibration: %d reads in %.2fs -> %d reads per step" % (nc, dt, ns))
        write_reads_fasta(sample_fa, buf, read_len, 0, ns)
        mini = max(1, int(math.ceil(ns * read_len / 3.0))) if ns * read_len < 3 * R.mo.mini_batch_size else None  # >= 3 mini-batches => the reference's read/map/write steps overlap
        times = []
        for it in range(a.warmup + a.steps):
            dt = R.map_file(sample_fa, sample_fa + ".ref.out", mini_batch=mini)
            if it >= a.warmup:
                times.append(dt)
        bases = paf_aligned_bases(sample_fa + ".ref.out", sam, ava)
        # single-thread figure on a small sample (per-core rate)
        n1 = min(ns, max(64, int(3e6 // read_len)))
        write_reads_fasta(sample_fa + ".t1", buf, read_len, 0, n1)
        dt1 = R.map_file(sample_fa + ".t1", sample_fa + ".t1.out", n_threads=1)
        b1 = paf_aligned_bases(sample_fa + ".t1.out", sam, ava)
        R.close()
        tot_t = sum(times)
        val = bases * len(times) / tot_t
        sample = ("%d of the %d reads per step (%d mini-batches of -K %s), same reference; mm_map_file() wall time incl. FASTA parsing and %s writing, "
                  "index build (%.0fs) excluded" % (ns, n_reads, 3 if mini else int(math.ceil(ns * read_len / R.mo.mini_batch_size)), mini or R.mo.mini_batch_size,
                                                   "SAM" if sam else "PAF", R.t_idx))
        line = {"metric": wl["metric"], "value": val, "unit": "bases/s", "n_gpus": a.gpus, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": 1e3 * tot_t / len(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "int8 DP cells (int32 scores), u64 hashes, f32 chain penalties", "data": "synthetic", "impl": "reference", "config": cfg,
                "cpu_baseline": {"value": val, "unit": "bases/s", "cores": n_threads_all, "logical_cpus": n_threads_all, "physical_cores": physical_cores(),
                                 "kind": "reference", "sample": sample, "sample_reads": ns,
                                 "t1": {"value": b1 / dt1, "unit": "bases/s", "cores": 1, "sample": "%d reads, -t 1" % n1}},
                "e2e": {"value": val, "unit": "bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # =====================================================================================================================
    # ---------------- this repo's arm ----------------
    al = make_aligner()
    qlens = np.full(n_reads, read_len, dtype=np.int32)
    prepared = al.prepare_batch(buf, qlens, names)

    def barrier():
        torch.cuda.synchronize()
        if dist_on:
            dist.barrier()
        torch.cuda.synchronize()

    dumped = {}

    def run_steps(n, resident, dump=False):
        L.mmb_set_resident_reads(1 if resident else 0)
        bases, times = 0, []
        for it in range(n):
            t = time.perf_counter()
            n_regs, regs, rep = al.map_prepared(prepared)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t)
            bases = int(L.mmb_aligned_bases(n_reads, n_regs.ctypes.data, regs.ctypes.data, 1 if wl["kind"] == "ava" else 0))
            if dump and it == n - 1:
                dumped.update(collect_outputs(api, n_regs, regs, rep))
            al.free_batch(n_regs, regs)
        return bases, times

    log("warm-up x%d" % a.warmup)
    run_steps(max(a.warmup, 3), True)
    try:
        free_b, tot_b = torch.cuda.mem_get_info()
        log("device memory after warm-up: %.1f of %.1f GB in use" % ((tot_b - free_b) / 1e9, tot_b / 1e9))
    except Exception:
        pass
    L.mmb_launch_count_all(1)
    sampler = ClockSampler(local_rank)
    sampler.start()
    try:
        # --- timed region A: `value` (read bases resident in HBM; only the mm_map_batch calls are timed) ---
        barrier()
        bases, times_a = run_steps(a.steps, True, dump=a.dump_outputs is not None)
        barrier()
        t_a = sum(times_a)
        launches = int(L.mmb_launch_count_all(0))
        # --- timed region B: `e2e` (host buffers in, results out) ---
        barrier()
        bases_b, times_b = run_steps(a.steps, False)
        barrier()
        t_b = sum(times_b)
        d2h_bytes = int(L.mmb_last_d2h_bytes())
    finally:  # the sampler is a child process: never leave it running
        clocks = sampler.stop()
    # --- timed region C (rank 0's own figure is reported; every rank runs it so that the host is loaded as in production):
    #     `file_e2e` = mm_map_file(): FASTA in (page cache), PAF/SAM out (tmpfs) -- what the reference arm's number contains ---
    file_e2e = None
    if not a.no_file_e2e:
        if wl["kind"] != "ava":
            write_reads_fasta(full_fa, buf, read_len, 0, n_reads)
        out_full = full_fa + ".out"
        tf = []
        barrier()
        for it in range(2):
            with StdoutTo(out_full):
                t = time.perf_counter()
                L.mm_map_file(al._idx, full_fa.encode(), C.byref(al.map_opt), nthr)
                C.CDLL(None).fflush(None)
                tf.append(time.perf_counter() - t)
        barrier()
        fb = paf_aligned_bases(out_full, sam, ava)
        file_e2e = {"value": fb / tf[-1], "unit": "bases/s", "ms_per_step": 1e3 * tf[-1], "per_gpu": True,
                    "what": "mm_map_file(): %d reads from FASTA (page cache) -> %s on tmpfs, second of two runs; reader / GPU scheduler / writer overlapped (map.cu)" % (n_reads, "SAM" if sam else "PAF"),
                    "in_bytes": os.path.getsize(full_fa), "out_bytes": os.path.getsize(out_full)}
        os.unlink(out_full)
    # --- per-kernel device time for the roofline: extra steps with the read groups serialised (one stream), so that
    #     CUDA-event durations are not inflated by kernels of other groups sharing the SMs ---
    L.mmb_set_groups(-int(os.environ.get("MM_B200_GROUPS", "12")))  # the default group count, run one after another
    L.mmb_profile_enable_all(1)
    for k in range(6):
        L.mmb_profile_ms_all(k, 1); L.mmb_profile_units_all(k, 1); L.mmb_profile_bytes_all(k, 1); L.mmb_profile_scopes_all(k, 1)
    n_prof = 2
    run_steps(n_prof, True)
    prof = {}
    for k, nm in enumerate(["sketch", "seed", "sort", "chain", "ksw", "other"]):
        prof[nm] = {"ms": L.mmb_profile_ms_all(k, 0), "units": int(L.mmb_profile_units_all(k, 0)), "bytes": int(L.mmb_profile_bytes_all(k, 0)),
                    "scopes": int(L.mmb_profile_scopes_all(k, 0))}
    L.mmb_profile_enable_all(0)
    L.mmb_set_groups(0)
    # max over ranks
    tt = torch.tensor([t_a, t_b], dtype=torch.float64, device="cuda")
    bb = torch.tensor([float(bases), float(bases_b)], dtype=torch.float64, device="cuda")
    if dist_on:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(bb, op=dist.ReduceOp.SUM)
    t_a, t_b = float(tt[0]), float(tt[1])
    tot_bases_a, tot_bases_b = float(bb[0]), float(bb[1])
    value = tot_bases_a * a.steps / t_a
    e2e = tot_bases_b * a.steps / t_b
    if rank != 0:
        if dist_on:
            dist.destroy_process_group()
        return 0
    # --- roofline of the dominant kernel (K3; for ava-ont, which runs no ksw2, the chaining stage) ---
    peak, peak_src = measured_peaks()
    dom = "ksw" if prof["ksw"]["ms"] > 0 else "chain"
    k = prof[dom]
    n_launch_k = max(1, k["scopes"])
    k_gbs = (k["bytes"] / 1e9) / (k["ms"] / 1e3) if k["ms"] > 0 else 0.0
    roofline = {"kernel": "K3 ksw2 kernels (ksw_pk_kernel + ksw_extd2_kernel)" if dom == "ksw" else "K2c chaining kernels (chain_fill + backtrack)",
                "bound": "hbm", "achieved": k_gbs, "peak": peak, "unit": "GB/s", "frac": k_gbs / peak,
                "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": k["bytes"] / n_launch_k, "avg_launch_ms": k["ms"] / n_launch_k,
                "stage_ms_per_step": {nm: prof[nm]["ms"] / n_prof for nm in prof},
                "timing": "CUDA events on the launch stream, %d profiled steps with the scheduler's read groups serialised" % n_prof}
    if dom == "ksw":
        roofline["gcups"] = (k["units"] / 1e9) / (k["ms"] / 1e3) if k["ms"] > 0 else 0.0
        roofline["note"] = ("integer-pipe bound by construction: ~%.0f DP cells per read base at 1 B/cell (traceback) algorithmic bytes; the HBM fraction is expected "
                            "to be small (SURVEY 8d)" % (k["units"] / max(1.0, tot_bases_a / max(1, world) * n_prof)))
    try:  # per-stage algorithmic bandwidth (DESIGN.md section 3 definitions); informational, never allowed to break the line
        roofline["stages"] = {nm: {"ms_per_step": prof[nm]["ms"] / n_prof, "algorithmic_gb_per_step": prof[nm]["bytes"] / n_prof / 1e9,
                                   "gb_per_s": (prof[nm]["bytes"] / 1e9) / (prof[nm]["ms"] / 1e3) if prof[nm]["ms"] > 0 else 0.0,
                                   "frac_of_hbm_peak": ((prof[nm]["bytes"] / 1e9) / (prof[nm]["ms"] / 1e3) / peak) if prof[nm]["ms"] > 0 and peak else 0.0}
                              for nm in ("sketch", "seed", "sort", "chain", "ksw")}
        roofline["stages"]["tail"] = {"ms_per_step": prof["other"]["ms"] / n_prof, "what": "K4 finalize_kernel (per-hit CIGAR assembly, mm_fix_cigar, mm_update_extra on the device) + ksw_ll probes"}
    except Exception:
        pass
    tp = os.path.join(ROOT, "profiles", "ksw_traffic.json")
    if dom == "ksw" and a.workload == "map-ont" and os.path.exists(tp):
        try:  # dram__bytes of the K3 launches from the committed `ncu --set full` capture of this command (profiles/README.md says which run)
            # the capture covers ONE alignment wave (all K3 kernels of one scheduler group); its DRAM bytes per algorithmic byte, times this
            # run's algorithmic bytes per launch set, is the per-launch figure (a launch set = one wave of one group, like `achieved`)
            tj = json.load(open(tp))
            roofline["traffic"] = tj["dram_bytes_wave"] / tj["algorithmic_bytes_wave"] * roofline["algorithmic_bytes_per_launch"]
            roofline["traffic_over_algorithmic"] = tj["dram_bytes_wave"] / tj["algorithmic_bytes_wave"]
            roofline["traffic_source"] = tj.get("source", "profiles/ksw_traffic.json")
        except Exception:
            pass
    line = {"metric": wl["metric"], "value": value, "unit": "bases/s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": 1e3 * t_a / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int8 DP cells (int32 scores), u64 hashes, f32 chain penalties", "data": "synthetic", "config": cfg,
            "host": {"threads_per_rank": nthr, "logical_cpus": n_threads_all, "physical_cores": physical_cores(), "pool_threads": int(os.environ["MM_B200_HOST_THREADS"])},
            "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": e2e, "unit": "bases/s", "ms_per_step": 1e3 * t_b / a.steps,
                    "h2d_bytes_per_step": int(n_reads * read_len + 12 * n_reads), "d2h_bytes_per_step": d2h_bytes},
            "roofline": roofline}
    if file_e2e:
        line["file_e2e"] = file_e2e
    if bcast:
        line["index_broadcast"] = bcast
    # --- CPU baseline + parity: the reference's own code on this box's cores, bounded sample, both arms through mm_map_file ---
    if not a.no_cpu_baseline:
        try:
            ns = min(a.cpu_sample or max(2000, int(2e8 // read_len)), n_reads)
            write_reads_fasta(sample_fa, buf, read_len, 0, ns)
            mini = max(1, int(math.ceil(ns * read_len / 3.0)))
            mo = api.MapOpt.from_buffer_copy(al.map_opt)
            mo.mini_batch_size = mini
            with StdoutTo(sample_fa + ".b200.out"):
                L.mm_map_file(al._idx, sample_fa.encode(), C.byref(mo), nthr)
                C.CDLL(None).fflush(None)
            if gidx is not None:
                log("writing the reference FASTA for the CPU baseline")
                L.mmb_idx_write_fasta(gidx, ref_fa.encode())
            mid_occ_mine = int(al.map_opt.mid_occ)
            al.close()
            gidx = None
            R = Reference(wl, ref_fa, n_threads_all, log)
            if R.ok:
                ct = R.map_file(sample_fa, sample_fa + ".ref.out", mini_batch=mini)
                cb = paf_aligned_bases(sample_fa + ".ref.out", sam, ava)
                n_ref, n_got, mism = compare_outputs(sample_fa + ".ref.out", sample_fa + ".b200.out", log, sam)
                line["parity"] = {"reads": ns, "ref_lines": n_ref, "b200_lines": n_got, "mismatches": mism, "mid_occ": [int(R.mo.mid_occ), mid_occ_mine],
                                  "what": "the same %d-read sample through mm_map_file() of both libraries, every %s record compared as text" % (ns, "SAM" if sam else "PAF")}
                n1 = min(ns, max(64, int(3e6 // read_len)))
                write_reads_fasta(sample_fa + ".t1", buf, read_len, 0, n1)
                dt1 = R.map_file(sample_fa + ".t1", sample_fa + ".t1.out", n_threads=1)
                b1 = paf_aligned_bases(sample_fa + ".t1.out", sam, ava)
                line["cpu_baseline"] = {"value": cb / ct, "unit": "bases/s", "cores": n_threads_all, "logical_cpus": n_threads_all, "physical_cores": physical_cores(),
                                        "kind": "reference",
                                        "sample": "%d of the %d reads of one step (3 mini-batches) vs the same reference; mm_map_file() wall %.2fs incl. parsing and output (index build %.0fs excluded)" % (ns, n_reads, ct, R.t_idx),
                                        "t1": {"value": b1 / dt1, "unit": "bases/s", "cores": 1, "sample": "%d reads, -t 1" % n1}}
                R.close()
        except Exception as e:  # the baseline is reported, never required for the GPU number
            line["cpu_baseline"] = {"value": None, "unit": "bases/s", "cores": n_threads_all, "kind": "reference", "sample": "failed: %r" % (e,)}
    if a.dump_outputs:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for nm, arr in dumped.items():
            np.save(os.path.join(a.dump_outputs, nm + ".npy"), arr)
    print(json.dumps(line))
    try:
        import shutil
        shutil.rmtree(tmp, ignore_errors=True)
    except Exception:
        pass
    if dist_on:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
