"""CPU: the whole product pipeline -- index build, sketch, seeding, sort, chaining, alignment kernels, scheduler, host logic, CLI --
compiled for the SIMT emulator of tests/cuda_emu (every CUDA kernel source unchanged, one OS thread per CUDA thread) and run on
the small golden cases; the output must equal the reference's recorded output byte for byte. Slow by nature (seconds per
kilobase), so only the small cases run here; the -m gpu suite covers everything on the real device."""
import os
import subprocess
import sys
import pytest
import oracle_lib as O

sys.path.insert(0, os.path.join(O.ROOT, "tests", "cuda_emu"))
GOLD = os.path.join(O.ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def emu_cli():
    import build_emu
    lib = build_emu.build("mmb_emu_all", build_emu.ALL, extra=())
    exe = os.path.join(os.path.dirname(lib), "minimap2-emu")
    main = os.path.join(O.ROOT, "minimap2_b200", "cli", "main.cc")
    if not os.path.exists(exe) or os.path.getmtime(exe) < max(os.path.getmtime(lib), os.path.getmtime(main)):
        subprocess.check_call(["g++", "-O1", "-I" + os.path.join(O.ROOT, "include"), "-o", exe, main, "-L" + os.path.dirname(lib), "-lmmb_emu_all",
                               "-Wl,-rpath,$ORIGIN", "-lpthread"])
    return exe


def cases():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLD, "make_golden.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m.CASES


GOLDEN = ["inv_paf_cigar", "x3s_paf_cigar", "t2_paf_cigar"]  # MT-human/MT-orang goes through the .mmi test below


def _splice_inputs(d, junc=False, spsc=False):
    """two cDNA reads, one per transcript strand; junc: no canonical signals in the genome, the introns come from a BED file instead"""
    import numpy as np
    import synth
    rng = np.random.default_rng(4)
    introns = []
    contigs = synth.random_genome(30_000, 33, n_contigs=1, repeat_frac=0.0)
    g = np.frombuffer(bytes(contigs[0]), dtype=np.uint8).copy()
    comp = np.zeros(256, dtype=np.uint8); comp[list(b"ACGT")] = list(b"TGCA")
    reads = []
    for i in range(2):
        pos = int(rng.integers(1000, len(g) - 6000)); exons = []; rev = i % 2 == 1
        for k in range(3):
            el = int(rng.integers(90, 200)); exons.append((pos, pos + el)); il = int(rng.integers(150, 500))
            d_, a_ = (b"GT", b"AG") if not rev else (b"CT", b"AC")
            if not junc and not spsc:
                g[pos + el:pos + el + 2] = list(d_); g[pos + el + il - 2:pos + el + il] = list(a_)
            if k < 2:
                introns.append((pos + el, pos + el + il, "-" if rev else "+"))
            pos += el + il
        tr = np.concatenate([g[s:e] for s, e in exons])
        reads.append(synth.mutate_ascii(comp[tr[::-1]] if rev else tr, rng, 0.03))
    tag = "spj" if junc else "sps" if spsc else "sp"
    rf, qf = os.path.join(d, tag + "_ref.fa"), os.path.join(d, tag + "_reads.fa")
    synth.write_fasta(rf, ["chr0"], [g.tobytes()]); synth.write_fasta(qf, ["tr0", "tr1"], reads)
    if spsc:  # splice-score file: contig, position, strand, D/A, score -- the true sites plus noise on both strands
        fn = os.path.join(d, "sps.txt")
        with open(fn, "w") as f:
            for st, en, sd in introns:
                dp, ap = (st, en - 1) if sd == "+" else (en - 1, st)
                f.write("chr0\t%d\t%s\tD\t%d\nchr0\t%d\t%s\tA\t%d\n" % (dp, sd, int(rng.integers(5, 15)), ap, sd, int(rng.integers(5, 15))))
            for _ in range(400):
                f.write("chr0\t%d\t%s\t%s\t%d\n" % (int(rng.integers(1, len(g) - 1)), "+-"[int(rng.integers(0, 2))], "DA"[int(rng.integers(0, 2))], int(rng.integers(-10, 8))))
        return ["-x", "splice", "-c", "--cs", "--spsc", fn, rf, qf]
    if junc:
        bed = os.path.join(d, "spj.bed")
        open(bed, "w").write("".join("chr0\t%d\t%d\tj%d\t0\t%s\n" % (st, en, i, sd) for i, (st, en, sd) in enumerate(introns)))
        return ["-x", "splice", "-c", "--cs", "--junc-bed", bed, rf, qf]
    return ["-x", "splice", "-c", "--cs", rf, qf]


def _high_occ_inputs(d):
    import numpy as np
    import synth
    rng = np.random.default_rng(11)
    g = np.frombuffer(bytes(synth.random_genome(9_000, 5)[0]), dtype=np.uint8).copy()
    unit = g[200:600].copy()
    for k in range(9):
        s = 900 + k * 800
        g[s:s + 400] = unit
        g[s + rng.integers(0, 400, 3)] = list(b"ACG")  # a few point differences between the copies
    reads = [synth.mutate_ascii(g[s:s + 1300], rng, 0.04) for s in (300, 2500, 5200)]
    rf, qf = os.path.join(d, "ho_ref.fa"), os.path.join(d, "ho_reads.fa")
    synth.write_fasta(rf, ["chr0"], [g.tobytes()]); synth.write_fasta(qf, ["r0", "r1", "r2"], reads)
    return ["-c", "-f", "3", "-e", "150", "-K", "1500", rf, qf]  # -K: two mini-batches through the overlapped read/map/write steps


def _rechain_inputs(d):
    """-f 3,50 with -e 0: reads that lie inside copies of a repeat lose every seed to the first cutoff (no chain, rep_len > 0) and
    are chained again with the second one (map.c:293-316); a read with unique flanks keeps its first-pass chains"""
    import numpy as np
    import synth
    rng = np.random.default_rng(12)
    g = np.frombuffer(bytes(synth.random_genome(9_000, 6)[0]), dtype=np.uint8).copy()
    unit = g[200:700].copy()
    for k in range(8):
        s = 1000 + k * 900
        g[s:s + 500] = unit
        g[s + rng.integers(0, 500, 2)] = list(b"AC")
    reads = [synth.mutate_ascii(g[1930:2370], rng, 0.03), synth.mutate_ascii(g[4620:5080], rng, 0.03), synth.mutate_ascii(g[5000:6500], rng, 0.04)]
    rf, qf = os.path.join(d, "rc_ref.fa"), os.path.join(d, "rc_reads.fa")
    synth.write_fasta(rf, ["chr0"], [g.tobytes()]); synth.write_fasta(qf, ["in0", "in1", "span"], reads)
    return ["-c", "-f", "3,50", "-e", "0", rf, qf]


def _qstrand_inputs(d):
    """--qstrand: reverse-strand hits are chained and aligned on the other strand of the target with the query kept forward"""
    import numpy as np
    import synth
    rng = np.random.default_rng(51)
    g = np.frombuffer(bytes(synth.random_genome(12_000, 23)[0]), dtype=np.uint8).copy()
    comp = np.zeros(256, dtype=np.uint8); comp[list(b"ACGT")] = list(b"TGCA")
    reads = [synth.mutate_ascii(g[800:2300], rng, 0.06), synth.mutate_ascii(comp[g[3000:4700][::-1]], rng, 0.06),
             synth.mutate_ascii(np.concatenate([comp[g[7000:7900][::-1]], comp[g[6100:6800][::-1]]]), rng, 0.04)]
    rf, qf = os.path.join(d, "qs_ref.fa"), os.path.join(d, "qs_reads.fa")
    synth.write_fasta(rf, ["chr0"], [g.tobytes()]); synth.write_fasta(qf, ["fwd", "rev", "rev_del"], reads)
    return ["-c", "--cs", "--qstrand", rf, qf]


def _sdust_inputs(d):
    """-T 20: query minimizers inside low-complexity stretches (microsatellites present many times in the genome) are masked
    before seeding (mm_dust_minier, map.c:33-57,68-69)"""
    import numpy as np
    import synth
    rng = np.random.default_rng(61)
    g = np.frombuffer(bytes(synth.random_genome(10_000, 29)[0]), dtype=np.uint8).copy()
    for st in (1500, 4200, 7700):  # the same microsatellite at three places
        g[st:st + 160] = np.frombuffer(b"ACACACACATACACACACGC" * 8, dtype=np.uint8)
    g[5600:5680] = ord("A")
    reads = [synth.mutate_ascii(g[900:2400], rng, 0.04), synth.mutate_ascii(g[3800:6000], rng, 0.05), synth.mutate_ascii(g[7650:7900], rng, 0.02)]
    rf, qf = os.path.join(d, "sd_ref.fa"), os.path.join(d, "sd_reads.fa")
    synth.write_fasta(rf, ["chr0"], [g.tobytes()]); synth.write_fasta(qf, ["r0", "r1", "r2"], reads)
    return ["-c", "-T", "20", "-w", "5", rf, qf]


def _many_waves_inputs(d):
    """a case the fuzzing tool found (seed 6017): with -z 30,20 a read keeps being split by z-drop and its alignment needs far more
    than 16 GPU waves -- the former fixed bound of the scheduler"""
    import importlib.util
    spec = importlib.util.spec_from_file_location("fuzz_cli", os.path.join(O.ROOT, "tests", "cuda_emu", "fuzz_cli.py"))
    fz = importlib.util.module_from_spec(spec); spec.loader.exec_module(fz)
    old = os.environ.get("DRY"); os.environ["DRY"] = "1"
    try:
        args = fz.one_(6017)[2].split()
    finally:
        if old is None:
            del os.environ["DRY"]
        else:
            os.environ["DRY"] = old
    return [a for a in args if a != "--qstrand"]


def _asm_inputs(d, preset, div):
    import numpy as np
    import synth
    rng = np.random.default_rng(21)
    g = np.frombuffer(bytes(synth.random_genome(24_000, 9)[0]), dtype=np.uint8).copy()
    comp = np.zeros(256, dtype=np.uint8); comp[list(b"ACGT")] = list(b"TGCA")
    if preset == "asm5":  # sparse seeds (w=19) and unpacked scoring make this the slow one under emulation: keep it short
        cs = [np.concatenate([g[1000:2100], g[2350:3300]]), comp[g[9000:10200][::-1]]]
    else:
        cs = [np.concatenate([g[1000:3200], g[3450:5200], comp[g[5200:6500][::-1]]]), g[9000:13500]]
    contigs = [synth.mutate_ascii(c, rng, div) for c in cs]
    rf, qf = os.path.join(d, preset + "_ref.fa"), os.path.join(d, preset + "_asm.fa")
    synth.write_fasta(rf, ["chr0"], [g.tobytes()]); synth.write_fasta(qf, ["ctg0", "ctg1"], contigs)
    return ["-x", preset, "-c", "--cs", rf, qf]


def _alt_inputs(d):
    import numpy as np
    import synth
    rng = np.random.default_rng(31)
    g = np.frombuffer(bytes(synth.random_genome(12_000, 13)[0]), dtype=np.uint8).copy()
    alt = np.frombuffer(synth.mutate_ascii(g[3000:7000], rng, 0.003), dtype=np.uint8)  # an ALT haplotype of chr0:3000-7000
    reads = [synth.mutate_ascii(alt[500:1900], rng, 0.05), synth.mutate_ascii(g[3600:5000], rng, 0.05), synth.mutate_ascii(g[8000:9200], rng, 0.05)]
    rf, qf, af = os.path.join(d, "alt_ref.fa"), os.path.join(d, "alt_reads.fa"), os.path.join(d, "alt.txt")
    synth.write_fasta(rf, ["chr0", "chr0_alt"], [g.tobytes(), alt.tobytes()]); synth.write_fasta(qf, ["r0", "r1", "r2"], reads)
    open(af, "w").write("chr0_alt\tsome comment\nnot_a_contig\n")
    return ["-c", "--alt", af, "--alt-drop", "0.2", rf, qf]


def _ava_inputs(d):
    import numpy as np
    import synth
    rng = np.random.default_rng(41)
    g = np.frombuffer(bytes(synth.random_genome(7_000, 19)[0]), dtype=np.uint8).copy()
    g[4200:4600] = g[600:1000]  # a repeat, so that some minimizers exceed the occurrence cutoff of the read index
    comp = np.zeros(256, dtype=np.uint8); comp[list(b"ACGT")] = list(b"TGCA")
    reads = []
    for i, s in enumerate(range(0, 5000, 1000)):
        x = g[s:s + 2000]
        reads.append(synth.mutate_ascii(comp[x[::-1]] if i % 2 else x, rng, 0.05))
    qf = os.path.join(d, "ava_reads.fa")
    synth.write_fasta(qf, ["rd%d" % i for i in (3, 0, 4, 1, 2)], reads)  # names out of order: the NO_DUAL name comparison matters
    return ["-x", "ava-ont", "-f", "2", qf, qf]


def _edge_inputs(d):
    """FASTQ (gzipped, comments, qualities) with reads that cannot map: shorter than k, all N, lower case, an N stretch"""
    import gzip
    import numpy as np
    import synth
    rng = np.random.default_rng(1)
    g = synth.random_genome(6000, 3)[0]
    r = np.frombuffer(bytes(g), dtype=np.uint8)
    reads = [("short", b"ACGTACGTAC"), ("allN", b"N" * 300), ("good", bytes(synth.mutate_ascii(r[1000:2200], rng, 0.05))),
             ("lower", bytes(synth.mutate_ascii(r[3000:3900], rng, 0.02)).lower()), ("withN", bytes(r[4000:4400]) + b"N" * 10 + bytes(r[4410:5000]))]
    rf, qf = os.path.join(d, "edge_ref.fa"), os.path.join(d, "edge_reads.fq.gz")
    synth.write_fasta(rf, ["chr0"], [bytes(g)])
    with gzip.open(qf, "wt") as f:
        for n, s_ in reads:
            f.write("@%s some comment\n%s\n+\n%s\n" % (n, s_.decode(), "I" * len(s_)))
    return ["-a", "-y", "-K", "1k", rf, qf]


def _multipart_inputs(d):
    """-I 4k splits a three-contig reference into several index parts; every part is mapped in turn (main.c:437-511)"""
    import numpy as np
    import synth
    rng = np.random.default_rng(2)
    cs = synth.random_genome(9000, 5, n_contigs=3)
    reads = [bytes(synth.mutate_ascii(np.frombuffer(bytes(c), dtype=np.uint8)[500:1800], rng, 0.05)) for c in cs]
    rf, qf = os.path.join(d, "mp_ref.fa"), os.path.join(d, "mp_reads.fa")
    synth.write_fasta(rf, ["c0", "c1", "c2"], [bytes(c) for c in cs]); synth.write_fasta(qf, ["q0", "q1", "q2"], reads)
    return ["-c", "-I", "4k", "--paf-no-hit", rf, qf]


@pytest.fixture(scope="module")
def emu_runs(emu_cli, tmp_path_factory):
    """Every emulated CLI run of this module, started together (6 at a time): the emulator spends most of its time in thread
    rendezvous, so the runs overlap well and the module's wall time is that of the longest chain rather than the sum."""
    from concurrent.futures import ThreadPoolExecutor
    d = str(tmp_path_factory.mktemp("emu_e2e"))
    env = dict(os.environ, MM_B200_GROUPS="1")
    data = os.path.join(GOLD, "data")
    jobs = {}
    for name in GOLDEN:
        jobs[name] = (cases()[name], data, None)
    jobs["cig_overflow"] = (cases()["x3s_paf_cigar"], data, None, {"MM_B200_CIG_SHIFT": "6"})
    jobs["job_chunks"] = (cases()["x3s_paf_cigar"], data, None, {"MM_B200_JOB_CHUNK": "7"})
    jobs["splice"] = (_splice_inputs(d), d, True)
    jobs["splice_junc"] = (_splice_inputs(d, junc=True), d, True)
    jobs["splice_spsc"] = (_splice_inputs(d, spsc=True), d, True)
    jobs["high_occ"] = (_high_occ_inputs(d), d, True)
    jobs["asm5"] = (_asm_inputs(d, "asm5", 0.004), d, True)
    jobs["asm20"] = (_asm_inputs(d, "asm20", 0.03), d, True)
    jobs["alt"] = (_alt_inputs(d), d, True)
    jobs["ava"] = (_ava_inputs(d), d, True)
    jobs["edge"] = (_edge_inputs(d), d, True)
    jobs["rechain"] = (_rechain_inputs(d), d, True)
    jobs["qstrand"] = (_qstrand_inputs(d), d, True)
    jobs["sdust"] = (_sdust_inputs(d), d, True)
    jobs["waves"] = (_many_waves_inputs(d), d, True)
    jobs["multipart"] = (_multipart_inputs(d), d, True)

    def one(item):
        name, (args, cwd, with_ref), more_env = item[0], item[1][:3], (item[1][3] if len(item[1]) > 3 else {})
        ref = None
        if with_ref:
            ref = O.ref_cli_lines(args, cwd)
        p = subprocess.run([emu_cli, "-t", "4"] + args, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=1800, env=dict(env, **more_env))
        return name, dict(rc=p.returncode, err=p.stderr.decode()[-2000:], out=p.stdout.decode().splitlines(), ref=ref)

    order = sorted(jobs.items(), key=lambda kv: {"waves": 0, "splice": 0, "splice_junc": 0, "splice_spsc": 0, "inv_paf_cigar": 1, "asm20": 2}.get(kv[0], 9))  # longest first
    with ThreadPoolExecutor(6) as ex:
        return dict(ex.map(one, order))


@pytest.mark.parametrize("name", GOLDEN)
def test_emulated_pipeline_matches_recorded_reference(emu_runs, name):
    r = emu_runs[name]
    assert r["rc"] == 0, r["err"]
    got = [l for l in r["out"] if not l.startswith("@PG")]
    exp = open(os.path.join(GOLD, "expected", name + ".txt")).read().splitlines()
    assert got == exp, (len(got), len(exp), [(a[:200], b[:200]) for a, b in zip(got, exp) if a != b][:2])


def test_emulated_cigar_arena_overflow_is_recovered(emu_runs):
    """the CIGAR arena estimate (qlen+tlen)/2+8 per job is a heuristic; MM_B200_CIG_SHIFT shrinks it 64-fold so that every wave overflows:
    the chunk is rerun with the size the kernels reported and the host staging buffer grows (it used to abort: ADVICE round 1)"""
    r = emu_runs["cig_overflow"]
    assert r["rc"] == 0, r["err"]
    exp = open(os.path.join(GOLD, "expected", "x3s_paf_cigar.txt")).read().splitlines()
    assert r["out"] == exp


def test_emulated_many_job_chunks(emu_runs):
    """an alignment wave larger than the device result buffers runs in chunks (2^20 jobs); MM_B200_JOB_CHUNK=7 forces dozens of chunks per
    wave: per-chunk CIGAR arenas, their device addresses in the job cache, and K4 stitching pieces that live in different arenas"""
    r = emu_runs["job_chunks"]
    assert r["rc"] == 0, r["err"]
    exp = open(os.path.join(GOLD, "expected", "x3s_paf_cigar.txt")).read().splitlines()
    assert r["out"] == exp


def test_emulated_spliced_mapping_matches_reference(emu_runs):
    """-x splice end to end under the emulator (spliced kernel variant + splice branches of the driver) against the reference binary:
    two small cDNA reads, one per transcript strand"""
    r = emu_runs["splice"]
    assert r["rc"] == 0, r["err"]
    assert O.assert_same_lines(r["out"], r["ref"]) == 2


def test_emulated_junction_annotation_matches_reference(emu_runs):
    """-x splice --junc-bed: mm_idx_bed_read on the index, the intron table on the device, junction flags derived per ksw_exts2 job
    in the kernel (mm_idx_bed_junc's window rule), for a genome without canonical splice signals"""
    r = emu_runs["splice_junc"]
    assert r["rc"] == 0, r["err"]
    assert O.assert_same_lines(r["out"], r["ref"]) == 2


def test_emulated_splice_scores_match_reference(emu_runs):
    """-x splice --spsc: mm_idx_spsc_read2 on the index, per-strand score tables on the device, junc[] bytes assembled per ksw_exts2
    job in the kernel (mm_idx_spsc_get's window rule), KSW_EZ_SPLICE_SCORE on every spliced call"""
    r = emu_runs["splice_spsc"]
    assert r["rc"] == 0, r["err"]
    assert O.assert_same_lines(r["out"], r["ref"]) == 2


def test_emulated_high_occurrence_seed_selection_matches_reference(emu_runs):
    """mm_seed_select (seed.c:56-96) on the device: a genome made mostly of copies of one 400 bp unit and -f 3 put most minimizers of
    every read above mid_occ, so the streak selection (heap of the lowest-occurrence seeds per stretch, max_max_occ cut, rep_len)
    decides which seeds are kept; -e 150 makes several seeds per stretch survive. Output equals the reference binary's."""
    r = emu_runs["high_occ"]
    assert r["rc"] == 0, r["err"]
    assert O.assert_same_lines(r["out"], r["ref"]) >= 3
    assert any("rl:i:" in l and "rl:i:0" not in l for l in r["out"])  # the selection really masked something


@pytest.mark.parametrize("preset", ["asm5", "asm20"])
def test_emulated_assembly_presets_match_reference(emu_runs, preset):
    """-x asm5 / asm20 (MM_F_RMQ: mg_lchain_rmq is the first chainer, map.c:275-276, followed by the bw_long re-chain of
    map.c:283-292; heavy gap costs, bw 1000/100000): two contigs against a small genome, one carrying a 250 bp deletion and a
    reverse-complemented tail. Output equals the reference binary's."""
    r = emu_runs[preset]
    assert r["rc"] == 0, r["err"]
    assert O.assert_same_lines(r["out"], r["ref"]) >= 2


def test_emulated_second_occurrence_cutoff_matches_reference(emu_runs):
    """-f INT,INT: the re-chaining pass of map.c:293-316 (seeds collected again with max_occ for reads left without a chain)"""
    r = emu_runs["rechain"]
    assert r["rc"] == 0, r["err"]
    O.assert_same_lines(r["out"], r["ref"])
    assert any(l.startswith("in0\t") for l in r["out"]) and any(l.startswith("in1\t") for l in r["out"])  # mapped thanks to the second pass


def test_emulated_query_strand_mode_matches_reference(emu_runs):
    """--qstrand end to end: anchors of reverse hits in other-strand coordinates (map.c:188-192), jobs that read the target
    complemented (MMB_JOB_T_COMP, universal kernel), flipped PAF coordinates and cs on that view (format.c:343-346,440-443)"""
    r = emu_runs["qstrand"]
    assert r["rc"] == 0, r["err"]
    O.assert_same_lines(r["out"], r["ref"])
    assert sum(l.split("\t")[4] == "-" for l in r["out"]) >= 2


def test_emulated_sdust_masking_matches_reference(emu_runs):
    """-T: symmetric DUST intervals from the host (hl_sdust), minimizers squeezed on the device before the occurrence filter"""
    r = emu_runs["sdust"]
    assert r["rc"] == 0, r["err"]
    assert O.assert_same_lines(r["out"], r["ref"]) >= 2


def test_emulated_many_alignment_waves_match_reference(emu_runs):
    """repeated z-drop splits: more replay / GPU waves than the scheduler used to allow (regression test for a fuzzing find)"""
    r = emu_runs["waves"]
    assert r["rc"] == 0, r["err"]
    assert O.assert_same_lines(r["out"], r["ref"]) >= 1


def test_emulated_alt_contigs_match_reference(emu_runs):
    """--alt (mm_idx_alt_read index.c:648-670, mm_mark_alt + the ALT-aware mm_hit_sort / mm_set_parent of hit.c:91-223 at
    map.c:321-324): reads from a region with an ALT haplotype; the ALT hits are down-weighted like the reference does."""
    r = emu_runs["alt"]
    assert r["rc"] == 0, r["err"]
    assert O.assert_same_lines(r["out"], r["ref"]) >= 4
    r0 = [l.split("\t") for l in r["out"] if l.startswith("r0\t")]  # sampled from the ALT haplotype, yet the primary contig wins with MAPQ 60
    assert r0[0][5] == "chr0" and r0[0][11] == "60" and "tp:A:P" in r0[0] and r0[1][5] == "chr0_alt" and "tp:A:S" in r0[1]


def test_emulated_all_vs_all_overlap_matches_reference(emu_runs):
    """-x ava-ont reads-vs-reads (skip_seed of map.c:78-100 with NO_DIAG / NO_DUAL on the device, occ_dist = 0 branch of the seed
    selection, ALL_CHAINS, no base-level alignment): five overlapping reads, alternating strands, names out of order"""
    r = emu_runs["ava"]
    assert r["rc"] == 0, r["err"]
    assert O.assert_same_lines(r["out"], r["ref"]) >= 4


@pytest.mark.parametrize("name,n_min", [("edge", 7), ("multipart", 3)])
def test_emulated_cli_edge_cases_match_reference(emu_runs, name, n_min):
    """unmappable reads, gzipped FASTQ with comments in SAM (-a -y), several mini-batches; a multi-part index with --paf-no-hit"""
    r = emu_runs[name]
    assert r["rc"] == 0, r["err"]
    assert O.assert_same_lines(r["out"], r["ref"]) >= n_min


def test_mmi_files_are_interchangeable(emu_cli, tmp_path):
    """mm_idx_dump / mm_idx_load (index.c:475-569): this library maps with an index file written by the reference (MT-human.ref.mmi,
    `minimap2 -d` of the reference) and with its own, both giving the recorded reference output (MT-human / MT-orang, the golden
    mt_paf_cigar case); where oracle/_ref is built, the reference also maps with the index written here"""
    data = os.path.join(GOLD, "data")
    exp = open(os.path.join(GOLD, "expected", "mt_paf_cigar.txt")).read().splitlines()
    mine, theirs = str(tmp_path / "mine.mmi"), os.path.join(data, "MT-human.ref.mmi")
    env = dict(os.environ, MM_B200_GROUPS="1")
    subprocess.run([emu_cli, "-t", "2", "-d", mine, os.path.join(data, "MT-human.fa")], check=True, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env)
    assert os.path.getsize(mine) == os.path.getsize(theirs)
    if os.path.exists(O.REF_BIN):
        out = subprocess.run([O.REF_BIN, "-t", "2", "-c", mine, os.path.join(data, "MT-orang.fa")], check=True, stdout=subprocess.PIPE, stderr=subprocess.PIPE).stdout.decode().splitlines()
        assert out == exp
    for idx in (theirs, mine):
        out = subprocess.run([emu_cli, "-t", "2", "-c", idx, os.path.join(data, "MT-orang.fa")], check=True, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env, timeout=1200).stdout.decode().splitlines()
        assert out == exp, idx


def test_emulated_spliced_extension_ignores_the_band(emu_cli):
    """ksw_exts2_sse takes no band (ksw2_exts2_sse.c:26-31). With -G 500 the driver's bandwidth (751) is smaller than the window of a right
    extension that runs on through a 766-bp intron; the spliced kernel used to clip the DP to that band and end the hit early (found by
    tests/cuda_emu/fuzz_cli.py --splice, seed 6009)."""
    data = os.path.join(GOLD, "data")
    args = ["-x", "splice", "-c", "--MD", "-C", "5", "-G", "500", os.path.join(data, "splice_G500_ref.fa"), os.path.join(data, "splice_G500_q.fa")]
    got = subprocess.run([emu_cli, "-t", "3"] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=dict(os.environ, MM_B200_GROUPS="1"), timeout=1200)
    assert got.returncode == 0, got.stderr.decode()[-1000:]
    out = got.stdout.decode().splitlines()
    O.assert_same_lines(out, O.ref_cli_lines(args))
    assert any("766N" in l for l in out)
