"""CPU: the seeding-stage restatement (oracle/mm2o_seed.c: index lookups, query-side filter, high-occurrence streak selection,
skip_seed, anchor expansion + radix sort) against the unmodified reference's own stage dump (`minimap2 --print-seeds`,
map.c:255-260): every anchor's contig, position, strand, query position and span, in order, and rep_len, for every read. The dump
is read from its recording under tests/golden/ref (per read: name, rep_len, anchor count and a digest of the anchor list)."""
import os
import subprocess
import numpy as np
import pytest
import oracle_lib as O
import synth


def sd_digest(sd):
    return O.line_digest("\n".join("%s\t%d\t%s\t%d\t%d" % a for a in sd))


def ref_seed_dump(args):
    def produce():
        p = subprocess.run([O.REF_BIN, "--print-seeds"] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
        assert p.returncode == 0, p.stderr.decode()[-1000:]
        reads, cur = [], None
        for l in p.stderr.decode().splitlines():
            f = l.split("\t")
            if f[0] == "QR":
                cur = dict(name=f[1], rep=None, sd=[]); reads.append(cur)
            elif f[0] == "RS":
                cur["rep"] = int(f[1])
            elif f[0] == "SD":
                cur["sd"].append((f[1], int(f[2]), f[3], int(f[4]), int(f[5])))
        return [dict(name=r["name"], rep=r["rep"], n_sd=len(r["sd"]), sd=sd_digest(r["sd"])) for r in reads]
    return O.recorded(["minimap2", "--print-seeds"] + O.cli_key(args), produce)


def oracle_seed_dump(idx, names, reads, qnames, **kw):
    out = []
    for s, qn in zip(reads, qnames):
        a, rep, _ = idx.anchors(s, qname=qn, **kw)
        sd = [(names[int(x << np.uint64(1) >> np.uint64(33))], int(np.int32(np.uint32(x & np.uint64(0xffffffff)))), "+-"[int(x >> np.uint64(63))],
               int(np.int32(np.uint32(y & np.uint64(0xffffffff)))), int(y >> np.uint64(32) & np.uint64(0xff))) for x, y in a]
        out.append(dict(name=qn, rep=rep, sd=sd))
    return out


def check(ref, mine):
    assert len(ref) == len(mine)
    for r, m in zip(ref, mine):
        assert r["name"] == m["name"] and r["rep"] == m["rep"], (r["name"], r["rep"], m["rep"])
        assert r["n_sd"] == len(m["sd"]), (r["name"], r["n_sd"], len(m["sd"]))
        assert r["sd"] == sd_digest(m["sd"]), (r["name"], m["sd"][:5])


@pytest.mark.parametrize("cfg", [dict(extra=["-f", "10"], kw=dict(mid_occ=10)),
                                 dict(extra=["-f", "6", "-e", "100"], kw=dict(mid_occ=6, occ_dist=100)),
                                 dict(extra=["-f", "8", "-e", "0"], kw=dict(mid_occ=8, occ_dist=0)),
                                 dict(extra=["-f", "10", "--q-occ-frac", "0"], kw=dict(mid_occ=10, q_occ_frac=0.0)),
                                 dict(extra=["-f", "10", "--for-only"], kw=dict(mid_occ=10, flag=0x100000)),
                                 dict(extra=["-f", "10", "--rev-only"], kw=dict(mid_occ=10, flag=0x200000))])
def test_seed_stage_vs_reference_dump(tmp_path, cfg):
    contigs = synth.random_genome(300_000, 5, n_contigs=3, repeat_frac=0.35)
    reads = synth.make_reads(contigs, 60, 3000, 0.08, 55, chimeric_frac=0.1)
    reads.append(contigs[0][1000:1400] * 6)  # a tandem-like read: the query-side multiplicity filter and tandem flags
    names = ["chr%d" % i for i in range(len(contigs))]
    qnames = ["read%d" % i for i in range(len(reads))]
    rf, qf = str(tmp_path / "ref.fa"), str(tmp_path / "reads.fa")
    synth.write_fasta(rf, names, contigs); synth.write_fasta(qf, qnames, reads)
    ref = ref_seed_dump(["-x", "map-ont"] + cfg["extra"] + [rf, qf])
    idx = O.OracleIndex([bytes(c) for c in contigs], names, 10, 15)
    check(ref, oracle_seed_dump(idx, names, [bytes(r) for r in reads], qnames, **cfg["kw"]))
    idx.close()


def test_seed_stage_all_vs_all(tmp_path):
    """-X: skip_seed's name tests (diagonal and dual overlaps) with the reads as their own reference"""
    contigs = synth.random_genome(120_000, 9, n_contigs=1, repeat_frac=0.1)
    reads = synth.make_reads(contigs, 70, 4000, 0.06, 99, chimeric_frac=0.0)
    qnames = ["rd%03d" % i for i in range(len(reads))]
    qf = str(tmp_path / "reads.fa")
    synth.write_fasta(qf, qnames, reads)
    ref = ref_seed_dump(["-x", "ava-ont", "-f", "20", qf, qf])
    idx = O.OracleIndex([bytes(r) for r in reads], qnames, 5, 15)
    mine = oracle_seed_dump(idx, qnames, [bytes(r) for r in reads], qnames, mid_occ=20, occ_dist=0, flag=0x001 | 0x002)
    check(ref, mine)
    idx.close()
