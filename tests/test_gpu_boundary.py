"""GPU: the drop-in boundary proven with the reference's OWN callers, unmodified, linked against libminimap2_b200.so
(tests/boundary/build_boundary.py, run by build() into oracle/_ref/boundary): example.c (mm_idx_reader_*, mm_mapopt_update, mm_tbuf_*, mm_map, kseq), main.c (the complete CLI incl.
mm_write_sam_hdr, mm_map_file) and the Cython binding mappy (python/mappy.pyx + cmappy.h: Aligner, map with cs/MD, ThreadBuffer, fastx_read,
seq, revcomp; several threads sharing one Aligner). Expected outputs were produced by the same callers linked against the reference library
(tests/golden/make_boundary_golden.py)."""
import json
import os
import subprocess
import sys
import pytest
import oracle_lib as O

pytestmark = pytest.mark.gpu
BUILD = os.path.join(O.ORACLE_DIR, "_ref", "boundary")
GOLD = os.path.join(O.ROOT, "tests", "golden")
DATA = os.path.join(GOLD, "data")
need = pytest.mark.skipif(not os.path.exists(os.path.join(BUILD, "example")), reason="oracle/_ref/boundary not built")


@need
def test_reference_example_c_runs_on_this_library():
    p = subprocess.run([os.path.join(BUILD, "example"), "MT-human.fa", "MT-orang.fa"], cwd=DATA, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert p.returncode == 0, p.stderr.decode()[-1500:]
    assert p.stdout.decode() == open(os.path.join(GOLD, "expected", "example_mt.txt")).read()


@need
@pytest.mark.parametrize("case", ["mt_sam", "mt_paf_cigar", "inv_paf_cigar"])
def test_reference_main_c_runs_on_this_library(case):
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLD, "make_golden.py"))
    m = importlib.util.module_from_spec(spec); spec.loader.exec_module(m)
    p = subprocess.run([os.path.join(BUILD, "minimap2-refmain"), "-t", "4"] + m.CASES[case], cwd=DATA, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert p.returncode == 0, p.stderr.decode()[-1500:]
    got = [l for l in p.stdout.decode().splitlines() if not l.startswith("@PG")]
    assert got == open(os.path.join(GOLD, "expected", case + ".txt")).read().splitlines()


@need
def test_reference_main_c_read_group():
    """-R: @RG header line with escapes resolved and RG:Z: on every record (format.c:82-117,639)"""
    p = subprocess.run([os.path.join(BUILD, "minimap2-refmain"), "-a", "-R", "@RG\\tID:grp1\\tSM:x", "MT-human.fa", "MT-orang.fa"], cwd=DATA,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert p.returncode == 0, p.stderr.decode()[-1500:]
    out = p.stdout.decode().splitlines()
    assert "@RG\tID:grp1\tSM:x" in out
    recs = [l for l in out if not l.startswith("@")]
    assert recs and all("\tRG:Z:grp1" in l for l in recs)
    exp = [l for l in open(os.path.join(GOLD, "expected", "mt_sam.txt")).read().splitlines() if not l.startswith("@")]
    assert [l.replace("\tRG:Z:grp1", "") for l in recs] == exp


@need
def test_reference_mappy_binding_runs_on_this_library():
    sys.path.insert(0, GOLD)
    import make_boundary_golden as G
    got = G.run_mappy(BUILD)
    exp = json.load(open(os.path.join(GOLD, "expected", "mappy_mt.json")))
    assert sorted(got) == sorted(exp)
    for k in exp:
        assert got[k] == exp[k], k
