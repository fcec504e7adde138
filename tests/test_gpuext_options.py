"""GPU parity for options OUTSIDE the hot-path scope table (SURVEY section 8): assembly presets (MM_F_RMQ as first chainer), --alt,
--junc-bed, --spsc, -f a,b, --qstrand, -T. They carry their own marker `gpu_ext` (NOT `gpu`) so that an optional feature can never
stop `pytest -m gpu -x` before an in-scope row; run them with `pytest -m gpu_ext`. CLI output vs the unmodified reference
binary, byte for byte."""
import os
import numpy as np
import pytest
import synth
from test_gpu_e2e import compare, DATA

pytestmark = pytest.mark.gpu_ext


@pytest.mark.parametrize("preset", ["asm5", "asm10", "asm20"])
def test_mt_assembly_presets(preset):
    compare(["-x", preset, "-c", "--cs", os.path.join(DATA, "MT-human.fa"), os.path.join(DATA, "MT-orang.fa")])


@pytest.mark.parametrize("preset,div", [("asm5", 0.003), ("asm10", 0.02), ("asm20", 0.05)])
def test_synthetic_contigs(tmp_path, preset, div):
    rng = np.random.default_rng(77)
    contigs = synth.random_genome(1_500_000, 31, n_contigs=2, repeat_frac=0.15)
    comp = np.zeros(256, dtype=np.uint8); comp[list(b"ACGT")] = list(b"TGCA")
    asm = []
    for i in range(24):  # contigs of 20-120 kb with a deletion, an insertion and sometimes an inverted segment
        c = np.frombuffer(bytes(contigs[i % 2]), dtype=np.uint8)
        L = int(rng.integers(20_000, 120_000)); s = int(rng.integers(0, len(c) - L))
        x = c[s:s + L]
        d0 = int(rng.integers(2000, L // 2)); dl = int(rng.integers(50, 3000))
        parts = [x[:d0], x[d0 + dl:L * 2 // 3], synth.ALPHA[rng.integers(0, 4, int(rng.integers(30, 1500)))], x[L * 2 // 3:]]
        if i % 3 == 0:
            parts[-1] = comp[parts[-1][::-1]]
        y = np.concatenate(parts)
        if i % 2:
            y = comp[y[::-1]]
        asm.append(synth.mutate_ascii(y, rng, div))
    rf, qf = str(tmp_path / "ref.fa"), str(tmp_path / "asm.fa")
    synth.write_fasta(rf, ["chr%d" % i for i in range(len(contigs))], contigs)
    synth.write_fasta(qf, ["ctg%d" % i for i in range(len(asm))], asm)
    n = compare(["-x", preset, "-c", "--cs", rf, qf])
    assert n >= len(asm)


def test_alt_contigs(tmp_path):
    """--alt / --alt-drop (index.c:648-670, hit.c:91-223, map.c:321-324): ALT haplotypes of several regions next to the primary contigs"""
    rng = np.random.default_rng(5)
    contigs = synth.random_genome(600_000, 51, n_contigs=2, repeat_frac=0.1)
    names = ["chr0", "chr1"]; seqs = [bytes(c) for c in contigs]; alts = []
    for i in range(6):
        c = np.frombuffer(seqs[i % 2], dtype=np.uint8)
        s = int(rng.integers(0, len(c) - 40_000)); L = int(rng.integers(8_000, 40_000))
        alts.append(synth.mutate_ascii(c[s:s + L], rng, [0.002, 0.01, 0.03][i % 3]))
        names.append("chr%d_alt%d" % (i % 2, i)); seqs.append(alts[-1])
    reads = synth.make_reads([np.frombuffer(x, dtype=np.uint8) for x in seqs], 400, 5000, 0.08, 77, chimeric_frac=0.03)
    rf, qf, af = str(tmp_path / "ref.fa"), str(tmp_path / "reads.fa"), str(tmp_path / "alt.txt")
    synth.write_fasta(rf, names, seqs)
    synth.write_fasta(qf, ["read%d" % i for i in range(len(reads))], reads)
    open(af, "w").write("".join(n + "\n" for n in names[2:]))
    n = compare(["-x", "map-ont", "-c", "--alt", af, rf, qf])
    assert n >= 400
    compare(["-x", "map-ont", "-a", "--alt", af, "--alt-drop", "0.3", rf, qf])


def test_junction_annotation_vs_reference(tmp_path):
    """-x splice --junc-bed (mm_idx_bed_read index.c:672-800; junction flags per ksw_exts2 call, align.c:638-643, derived in the
    kernel from the device intron table with mm_idx_bed_junc's window rule): transcripts over a genome where only a third of the
    introns carry canonical signals, annotation with duplicates, shifted decoys and both strands"""
    from test_aligndriver_vs_ref import _spliced_set, _write_bed
    rng = np.random.default_rng(15)
    g, reads, introns = _spliced_set(70, 150, glen=800_000)
    rf, qf, bed = str(tmp_path / "ref.fa"), str(tmp_path / "reads.fa"), str(tmp_path / "anno.bed")
    synth.write_fasta(rf, ["chr0"], [g]); synth.write_fasta(qf, ["tr%d" % i for i in range(len(reads))], reads)
    _write_bed(bed, introns, rng)
    assert compare(["-x", "splice", "-c", "--cs", "--junc-bed", bed, rf, qf]) >= 120
    compare(["-x", "splice", "--junc-bed", bed, "--junc-bonus", "5", "-a", rf, qf])


def test_splice_kernel_with_junction_table_matches_oracle():
    """the same check as tests/test_emu_ksw.py::test_emulated_splice_kernel_with_junction_annotation on the device, 200 jobs per model"""
    import ctypes as C
    import minimap2_b200 as mb
    from minimap2_b200._lib import KswJob, KswRes, KswScore, lib
    import test_emu_ksw as E
    L = lib()
    L.mmb_ctx_set_junctions.restype = C.c_int
    L.mmb_ctx_set_junctions.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    ctx = mb.Context(0)
    E.check_splice_jobs((L, C.c_void_p(ctx.h), KswJob, KswRes, KswScore), np.random.default_rng(179), (0x400 | 0x800, 0x400, 0), 200, 5, with_junc=True)
    ctx.close()


@pytest.mark.parametrize("extra", [["-f", "4,400", "-e", "0"], ["-f", "8,2000"]])
def test_second_occurrence_cutoff(tmp_path, extra):
    """-f INT,INT (map.c:293-316): reads left without a chain by the first cutoff collect their seeds again with the second one"""
    contigs = synth.random_genome(400_000, 61, n_contigs=2, repeat_frac=0.6)
    reads = synth.make_reads(contigs, 500, 1500, 0.06, 161, chimeric_frac=0.0)
    rf, qf = str(tmp_path / "ref.fa"), str(tmp_path / "reads.fa")
    synth.write_fasta(rf, ["chr%d" % i for i in range(len(contigs))], contigs)
    synth.write_fasta(qf, ["read%d" % i for i in range(len(reads))], reads)
    compare(["-c"] + extra + [rf, qf])


def test_splice_scores_vs_reference(tmp_path):
    """-x splice --spsc (mm_idx_spsc_read2 / mm_idx_spsc_get, index.c:963-1075; KSW_EZ_SPLICE_SCORE, align.c:688)"""
    from test_aligndriver_vs_ref import _spliced_set, _write_spsc
    rng = np.random.default_rng(16)
    g, reads, introns = _spliced_set(71, 150, glen=800_000)
    rf, qf, fn = str(tmp_path / "ref.fa"), str(tmp_path / "reads.fa"), str(tmp_path / "sc.txt")
    synth.write_fasta(rf, ["chr0"], [g]); synth.write_fasta(qf, ["tr%d" % i for i in range(len(reads))], reads)
    _write_spsc(fn, g, introns, rng)
    assert compare(["-x", "splice", "-c", "--cs", "--spsc", fn, rf, qf]) >= 120
    compare(["-x", "splice", "--spsc", fn, "--spsc-scale", "1", "--spsc0", "3", "-a", rf, qf])


def test_splice_kernel_with_score_tables_matches_oracle():
    """tests/test_emu_ksw.py::test_emulated_splice_kernel_with_splice_scores on the device, 200 jobs per model"""
    import ctypes as C
    import minimap2_b200 as mb
    from minimap2_b200._lib import KswJob, KswRes, KswScore, lib
    import test_emu_ksw as E
    L = lib()
    L.mmb_ctx_set_splice_scores.restype = C.c_int
    L.mmb_ctx_set_splice_scores.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]
    ctx = mb.Context(0)
    E.check_splice_jobs((L, C.c_void_p(ctx.h), KswJob, KswRes, KswScore), np.random.default_rng(181), (0x400 | 0x800, 0x400, 0), 200, 5, with_score=True)
    ctx.close()


def test_query_strand_mode(tmp_path):
    """--qstrand (main.c:252; map.c:188-192; align.c:780-783,815-818,875-878,899-901; format.c:343-346,440-443)"""
    contigs = synth.random_genome(500_000, 71, n_contigs=2, repeat_frac=0.1)
    reads = synth.make_reads(contigs, 300, 4000, 0.08, 171, chimeric_frac=0.05)
    rf, qf = str(tmp_path / "ref.fa"), str(tmp_path / "reads.fa")
    synth.write_fasta(rf, ["chr%d" % i for i in range(len(contigs))], contigs)
    synth.write_fasta(qf, ["read%d" % i for i in range(len(reads))], reads)
    assert compare(["-x", "map-ont", "-c", "--cs", "--qstrand", rf, qf]) >= 280
    compare(["--qstrand", rf, qf])


def test_sdust_masking(tmp_path):
    """-T 20 (mm_dust_minier, map.c:33-57): reads over a genome seeded with microsatellites and homopolymer runs"""
    rng = np.random.default_rng(17)
    contigs = synth.random_genome(400_000, 81, n_contigs=2, repeat_frac=0.05)
    gs = [np.frombuffer(bytes(c), dtype=np.uint8).copy() for c in contigs]
    for g in gs:
        for _ in range(150):
            st = int(rng.integers(0, len(g) - 400)); unit = synth.ALPHA[rng.integers(0, 4, int(rng.integers(1, 5)))]
            L = int(rng.integers(40, 300)); g[st:st + L] = np.resize(unit, L)
    reads = synth.make_reads(gs, 300, 3000, 0.06, 181, chimeric_frac=0.02)
    rf, qf = str(tmp_path / "ref.fa"), str(tmp_path / "reads.fa")
    synth.write_fasta(rf, ["chr0", "chr1"], [g.tobytes() for g in gs])
    synth.write_fasta(qf, ["read%d" % i for i in range(len(reads))], reads)
    assert compare(["-c", "-T", "20", rf, qf]) >= 280
    compare(["-x", "map-ont", "-T", "12", rf, qf])


def test_spliced_extension_ignores_the_band():
    """-x splice -G 500: the driver's bandwidth (751) is narrower than the window of a right extension that runs on through a 766-bp intron;
    ksw_exts2_sse takes no band (ksw2_exts2_sse.c:26-31). Device counterpart of tests/test_emu_e2e.py::test_emulated_spliced_extension_ignores_the_band
    (added after the round's last device session: first device run pending)."""
    n = compare(["-x", "splice", "-c", "--MD", "-C", "5", "-G", "500", os.path.join(DATA, "splice_G500_ref.fa"), os.path.join(DATA, "splice_G500_q.fa")])
    assert n == 3
