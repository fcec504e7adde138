"""GPU end-to-end parity: the B200 mapper's CLI output vs the unmodified reference binary (oracle/_ref/minimap2) on the
same inputs -- every PAF column and tag (NM ms AS nn tp cm s1 s2 de/dv zd rl cg) must match byte for byte. The reference's
output is read from its recording under tests/golden/ref (oracle_lib.recorded)."""
import os
import subprocess
import numpy as np
import pytest
import oracle_lib as O
import synth

pytestmark = pytest.mark.gpu
ROOT = O.ROOT
MINE = os.path.join(ROOT, "minimap2_b200", "minimap2-b200")
DATA = os.path.join(ROOT, "tests", "golden", "data")


def run(binary, args):
    p = subprocess.run([binary] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=1200)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    return p.stdout.decode().splitlines()


def compare(args):
    return O.assert_same_lines(run(MINE, ["-t", "8"] + args), O.ref_cli_lines(args))


def test_mt_paf():
    assert compare(["-c", os.path.join(DATA, "MT-human.fa"), os.path.join(DATA, "MT-orang.fa")]) == 1


def test_mt_sam_config0():
    """BASELINE.json configs[0]: minimap2 -a test/MT-human.fa test/MT-orang.fa"""
    compare(["-a", os.path.join(DATA, "MT-human.fa"), os.path.join(DATA, "MT-orang.fa")])


def test_mt_nocigar():
    compare([os.path.join(DATA, "MT-human.fa"), os.path.join(DATA, "MT-orang.fa")])


def test_inversion_pair():
    assert compare(["-c", os.path.join(DATA, "t-inv.fa"), os.path.join(DATA, "q-inv.fa")]) == 6


@pytest.mark.parametrize("cfg", [dict(seed=1, glen=2_000_000, n=300, rlen=10000, err=0.10, rep=0.0, chim=0.0),
                                 dict(seed=2, glen=1_000_000, n=200, rlen=8000, err=0.12, rep=0.2, chim=0.1),
                                 dict(seed=3, glen=500_000, n=300, rlen=3000, err=0.05, rep=0.1, chim=0.05)])
def test_synthetic_map_ont(tmp_path, cfg):
    contigs = synth.random_genome(cfg["glen"], cfg["seed"], n_contigs=3, repeat_frac=cfg["rep"])
    reads = synth.make_reads(contigs, cfg["n"], cfg["rlen"], cfg["err"], cfg["seed"] + 100, chimeric_frac=cfg["chim"])
    rf, qf = str(tmp_path / "ref.fa"), str(tmp_path / "reads.fa")
    synth.write_fasta(rf, ["chr%d" % i for i in range(len(contigs))], contigs)
    synth.write_fasta(qf, ["read%d" % i for i in range(len(reads))], reads)
    n = compare(["-x", "map-ont", "-c", "--cs", rf, qf])
    assert n >= cfg["n"] * 0.9


@pytest.mark.parametrize("gap", [["-O4", "-E2"], ["-O6", "-E3"]])
def test_single_affine_gap_cost(tmp_path, gap):
    """q == q2 and e == e2 select ksw_extz2 in the reference (align.c:360); here the dual-affine kernels run with equal terms"""
    compare(["-c"] + gap + [os.path.join(DATA, "MT-human.fa"), os.path.join(DATA, "MT-orang.fa")])
    contigs = synth.random_genome(400_000, 21, n_contigs=2, repeat_frac=0.1)
    reads = synth.make_reads(contigs, 150, 4000, 0.10, 121, chimeric_frac=0.05)
    rf, qf = str(tmp_path / "ref.fa"), str(tmp_path / "reads.fa")
    synth.write_fasta(rf, ["chr%d" % i for i in range(len(contigs))], contigs)
    synth.write_fasta(qf, ["read%d" % i for i in range(len(reads))], reads)
    compare(["-x", "map-ont", "-c"] + gap + [rf, qf])


def _overlap_set(tmp_path, seed, glen=300_000, n=240, rlen=5000):
    contigs = synth.random_genome(glen, seed, n_contigs=1, repeat_frac=0.05)
    reads = synth.make_reads(contigs, n, rlen, 0.08, seed + 7, chimeric_frac=0.0)
    qf = str(tmp_path / "reads.fa")
    synth.write_fasta(qf, ["rd%03d" % i for i in range(len(reads))], reads)
    return qf


def test_ava_ont_overlaps(tmp_path):
    """BASELINE config 4 shape: all-vs-all overlap, skip_seed's name tests (NO_DIAG, NO_DUAL) evaluated on the device"""
    qf = _overlap_set(tmp_path, 31)
    assert compare(["-x", "ava-ont", qf, qf]) > 100


def test_ava_with_cigar(tmp_path):
    """-X with base-level alignment: self-chain anchors carry MM_SEED_SELF into mm_align1 (align.c:760)"""
    qf = _overlap_set(tmp_path, 32, glen=150_000, n=100, rlen=4000)
    compare(["-x", "map-ont", "-X", "-c", qf, qf])


@pytest.mark.parametrize("strand", ["--for-only", "--rev-only"])
def test_strand_restricted(tmp_path, strand):
    compare(["-c", strand, os.path.join(DATA, "MT-human.fa"), os.path.join(DATA, "MT-orang.fa")])
    contigs = synth.random_genome(300_000, 41, n_contigs=2, repeat_frac=0.1)
    reads = synth.make_reads(contigs, 120, 4000, 0.10, 141, chimeric_frac=0.05)
    rf, qf = str(tmp_path / "ref.fa"), str(tmp_path / "reads.fa")
    synth.write_fasta(rf, ["chr%d" % i for i in range(len(contigs))], contigs)
    synth.write_fasta(qf, ["read%d" % i for i in range(len(reads))], reads)
    compare(["-x", "map-ont", "-c", strand, rf, qf])


@pytest.mark.parametrize("cfg", [dict(opts=["-x", "map-ont", "-c"], glen=20_000_000, n=1500, rlen=8000, err=0.10, rep=0.1, chim=0.05),
                                 dict(opts=["-x", "map-hifi", "-a"], glen=20_000_000, n=1000, rlen=12000, err=0.005, rep=0.1, chim=0.02),
                                 dict(opts=["-x", "ava-ont"], glen=1_500_000, n=800, rlen=6000, err=0.08, rep=0.0, chim=0.0)])
def test_scheduler_scale(tmp_path, cfg):
    """Batches large enough (>= 768 reads and >= 4 Mbases) for the scheduler to cut them into its 12 concurrent read groups -- the
    configuration the benchmark runs in: per-group streams and arenas, the device-slot gate, the shared host pool, K4 per group.
    Every output line must still equal the reference's, in input order."""
    contigs = synth.random_genome(cfg["glen"], 11, n_contigs=5, repeat_frac=cfg["rep"])
    reads = synth.make_reads(contigs, cfg["n"], cfg["rlen"], cfg["err"], 211, chimeric_frac=cfg["chim"])
    rf, qf = str(tmp_path / "ref.fa"), str(tmp_path / "reads.fa")
    synth.write_fasta(rf, ["chr%d" % i for i in range(len(contigs))], contigs)
    synth.write_fasta(qf, ["read%d" % i for i in range(len(reads))], reads)
    args = cfg["opts"] + ([qf, qf] if cfg["opts"][-1] == "ava-ont" else [rf, qf])
    assert O.assert_same_lines(run(MINE, ["-t", "16"] + args), O.ref_cli_lines(args)) >= cfg["n"] * 0.5
