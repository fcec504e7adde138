"""GPU parity of the spliced-alignment path (-x splice: the ksw_exts2 variant of the universal kernel + the splice branches of the
driver). The path was validated before its first device run by the SIMT emulator (tests/test_emu_ksw.py, tests/test_emu_e2e.py)
and by the CPU driver test (tests/test_aligndriver_vs_ref.py); these are the device-side checks. The file name sorts last on purpose."""
import os
import subprocess
import numpy as np
import pytest
import oracle_lib as O
import synth
from test_gpu_e2e import compare
from test_gpu_golden import load_cases, GOLD, MINE

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", sorted(k for k in load_cases().keys() if k.startswith("splice")))
def test_spliced_cli_output_matches_recorded_reference(name):
    args = load_cases()[name]
    p = subprocess.run([MINE, "-t", "8"] + args, cwd=os.path.join(GOLD, "data"), stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    got = [l for l in p.stdout.decode().splitlines() if not l.startswith("@PG")]
    exp = open(os.path.join(GOLD, "expected", name + ".txt")).read().splitlines()
    assert got == exp, [(a[:300], b[:300]) for a, b in zip(got, exp) if a != b][:2]


def test_splice_kernel_matches_oracle():
    """ksw_exts2 jobs through the C-ABI vs the oracle restatement (shared-memory tiers)"""
    import minimap2_b200 as mb
    from minimap2_b200 import kernels as K
    from test_emu_ksw import small_spliced_pair
    ctx = mb.Context(0)
    rng = np.random.default_rng(177)
    mat = O.simple_mat(1, 2, 1)
    for model in (0x400 | 0x800, 0x400, 0):
        pairs, params = [], []
        for it in range(200):
            q, t = small_spliced_pair(rng, int(rng.integers(1, 6)), float(rng.choice([0.0, 0.03, 0.1])))
            base = int(rng.choice([0, 0x08, 0x40, 0x40 | 0x02 | 0x80, 0x02]))
            pairs.append((q, t))
            params.append(dict(w=-1, zdrop=int(rng.choice([-1, 200])), end_bonus=int(rng.choice([-1, 10])), flag=base | int(rng.choice([0x100, 0x200])) | model | 0x80000))
        got = K.ksw_batch(ctx, K.make_score(mat, 2, 1, 32, 0, 9, 9, 5), pairs, params)
        for i, ((q, t), pr) in enumerate(zip(pairs, params)):
            exp = O.oracle_exts2(q, t, mat, 2, 1, 32, 9, pr["zdrop"], pr["end_bonus"], 9, 5, pr["flag"] & 0x1fff)
            assert got[i] == exp, (hex(model), i, len(q), len(t), hex(pr["flag"]))
    ctx.close()


def test_spliced_reads_vs_reference(tmp_path):
    """cDNA reads with introns up to 20 kb (the long ones run in the HBM-state tier), both transcript strands"""
    rng = np.random.default_rng(8)
    contigs = synth.random_genome(600_000, 43, n_contigs=2, repeat_frac=0.02)
    gs = [np.frombuffer(bytes(c), dtype=np.uint8).copy() for c in contigs]
    comp = np.zeros(256, dtype=np.uint8); comp[list(b"ACGT")] = list(b"TGCA")
    reads = []
    for i in range(120):
        g = gs[i % 2]
        pos = int(rng.integers(2000, len(g) - 120000)); exons = []; rev = i % 2 == 1
        for k in range(int(rng.integers(2, 7))):
            el = int(rng.integers(80, 400)); exons.append((pos, pos + el))
            il = int(rng.integers(100, 20000)) if k % 3 == 2 else int(rng.integers(100, 3000))
            if i % 4 != 3:
                d, a = (b"GT", b"AG") if not rev else (b"CT", b"AC")
                g[pos + el:pos + el + 2] = list(d); g[pos + el + il - 2:pos + el + il] = list(a)
            pos += el + il
        tr = np.concatenate([g[s:e] for s, e in exons])
        if rev:
            tr = comp[tr[::-1]]
        reads.append(synth.mutate_ascii(tr, rng, 0.03))
    rf, qf = str(tmp_path / "ref.fa"), str(tmp_path / "reads.fa")
    synth.write_fasta(rf, ["chr0", "chr1"], [g.tobytes() for g in gs])
    synth.write_fasta(qf, ["tr%d" % i for i in range(len(reads))], reads)
    assert compare(["-x", "splice", "-c", "--cs", rf, qf]) >= 100
    compare(["-x", "splice", "-uf", "-a", rf, qf])
