"""Pins the oracle (oracle/*.c) against the UNMODIFIED reference build (oracle/_ref, compiled from /root/reference).
CPU only. Skipped when oracle/_ref has not been built (it is built by __graft_entry__.build() in the dev container)."""
import ctypes as C
import numpy as np
import pytest
import oracle_lib as O

pytestmark = pytest.mark.skipif(not O.have_ref(), reason="oracle/_ref not built")

EXT, RIGHT, REVC, APPROX, GENERIC = 0x40, 0x02, 0x80, 0x08, 0x04


def rand_pair(rng, qlen, err):
    t = rng.integers(0, 4, qlen + rng.integers(0, 30)).astype(np.uint8)
    q = O.mutate(t, rng, err=err)
    if len(q) == 0:
        q = np.array([0], dtype=np.uint8)
    return q, t


@pytest.mark.parametrize("seed", range(6))
def test_extd2_matches_reference(seed):
    rng = np.random.default_rng(100 + seed)
    mat = O.simple_mat(2, 4, 1)
    n = 0
    for it in range(120):
        qlen = int(rng.integers(1, 400))
        q, t = rand_pair(rng, qlen, err=float(rng.choice([0.0, 0.05, 0.15, 0.4])))
        if rng.random() < 0.2:  # sprinkle N
            q[rng.integers(0, len(q))] = 4
            t[rng.integers(0, len(t))] = 4
        if rng.random() < 0.15:  # unrelated tail to trigger z-drop
            q = np.concatenate([q, rng.integers(0, 4, 300).astype(np.uint8)])
            t = np.concatenate([t, rng.integers(0, 4, 300).astype(np.uint8)])
        w = int(rng.choice([-1, 5, 17, 40, 100, 751, 30001]))
        zdrop = int(rng.choice([-1, 50, 200, 400]))
        eb = int(rng.choice([-1, 0, 10]))
        flag = int(rng.choice([0, APPROX, EXT, EXT | RIGHT | REVC, RIGHT, EXT | RIGHT, APPROX | RIGHT]))
        a = O.oracle_extd2(q, t, mat, 4, 2, 24, 1, w, zdrop, eb, flag)
        b = O.ref_extd2(q, t, mat, 4, 2, 24, 1, w, zdrop, eb, flag)
        assert a == b, (it, len(q), len(t), w, zdrop, eb, flag)
        n += 1
    assert n == 120


def test_extd2_other_scoring_and_generic():
    rng = np.random.default_rng(7)
    for (a_, b_, q, e, q2, e2, ts) in [(1, 4, 6, 2, 26, 1, 0), (1, 19, 39, 3, 81, 1, 0), (2, 6, 10, 2, 50, 1, 4), (1, 2, 2, 1, 32, 0, 0)]:
        mat = O.simple_mat(a_, b_, 1, ts)
        for it in range(40):
            qq, tt = rand_pair(rng, int(rng.integers(1, 300)), err=0.1)
            w = int(rng.choice([-1, 20, 200, 30001]))
            flag = int(rng.choice([0, APPROX, EXT, EXT | RIGHT | REVC]))
            if ts:
                flag |= GENERIC
            x = O.oracle_extd2(qq, tt, mat, q, e, q2, e2, w, 200, -1, flag)
            y = O.ref_extd2(qq, tt, mat, q, e, q2, e2, w, 200, -1, flag)
            assert x == y, (a_, b_, it, w, flag)


def test_extd2_long_band_limited():
    """end-extension shape: long sequences, w=751 so the band limits st0/en0 and 16-lane edge artefacts are live"""
    rng = np.random.default_rng(11)
    mat = O.simple_mat(2, 4, 1)
    for it in range(6):
        t = rng.integers(0, 4, 2500).astype(np.uint8)
        q = O.mutate(t, rng, err=0.12)
        for flag in (EXT, EXT | RIGHT | REVC, 0):
            for w in (751, 100, 33):
                x = O.oracle_extd2(q, t, mat, 4, 2, 24, 1, w, 400, -1, flag)
                y = O.ref_extd2(q, t, mat, 4, 2, 24, 1, w, 400, -1, flag)
                assert x == y, (it, flag, w)


def test_ll_i16():
    rng = np.random.default_rng(3)
    mat = O.simple_mat(2, 4, 1)
    for it in range(300):
        qq, tt = rand_pair(rng, int(rng.integers(1, 200)), err=float(rng.choice([0.0, 0.1, 0.3])))
        if rng.random() < 0.3:
            tt = np.concatenate([rng.integers(0, 4, int(rng.integers(0, 50))).astype(np.uint8), tt])
        assert O.oracle_ll_i16(qq, tt, mat, 4, 2) == O.ref_ll_i16(qq, tt, mat, 4, 2), it


@pytest.mark.parametrize("w,k,hpc", [(10, 15, 0), (5, 15, 0), (19, 19, 0), (10, 14, 0), (11, 21, 0), (10, 19, 1), (3, 4, 0), (50, 28, 0)])
def test_sketch(w, k, hpc):
    rng = np.random.default_rng(w * 100 + k)
    for it in range(60):
        n = int(rng.integers(1, 3000))
        alphabet = rng.choice([b"ACGT", b"ACGTN", b"AT", b"ACGTacgtNn", b"AC"])
        s = bytes(rng.choice(list(alphabet), n).astype(np.uint8))
        if rng.random() < 0.3:  # low complexity stretch
            s = s[: n // 2] + b"AT" * 40 + b"A" * 30 + s[n // 2:]
        a = O.oracle_sketch(s, w, k, rid=it, is_hpc=hpc)
        b = O.ref_sketch(s, w, k, rid=it, is_hpc=hpc)
        assert a.shape == b.shape and (a == b).all(), (it, n)


def test_radix_sort_tie_order():
    rng = np.random.default_rng(5)
    for it in range(200):
        n = int(rng.integers(0, 3000))
        bits = int(rng.choice([2, 6, 12, 20, 40, 64]))
        x = rng.integers(0, 2 ** min(bits, 63), n, dtype=np.uint64)
        if bits == 64:
            x = x * np.uint64(2) + rng.integers(0, 2, n, dtype=np.uint64)
        a = np.stack([x, np.arange(n, dtype=np.uint64)], axis=1)
        assert (O.oracle_sort128(a) == O.ref_sort128(a)).all(), it


def make_anchors(rng, n_chain=3, n_noise=200, qlen=10000, span=15):
    """anchors: x = rev<<63|rid<<32|rpos, y = span<<32|qpos; sorted by x with the oracle's radix sort (the reference's tie order:
    test_sort128 and the recorded vectors of tests/test_golden.py pin it), so that callers need no reference build"""
    rows = []
    for c in range(n_chain):
        rid = int(rng.integers(0, 3)); rev = int(rng.integers(0, 2))
        r0 = int(rng.integers(1000, 100000)); q = int(rng.integers(20, 200)); r = r0
        while q < qlen - 50:
            rows.append(((rev << 63) | (rid << 32) | r, (span << 32) | q))
            if rng.random() < 0.1:  # duplicate ref position (tie in x)
                rows.append(((rev << 63) | (rid << 32) | r, (span << 32) | (q + int(rng.integers(1, 30)))))
            step = int(rng.integers(1, 120))
            q += step; r += step + int(rng.integers(-6, 7)) * int(rng.random() < 0.3)
    for _ in range(n_noise):
        rows.append(((int(rng.integers(0, 2)) << 63) | (int(rng.integers(0, 3)) << 32) | int(rng.integers(0, 200000)),
                     (span << 32) | int(rng.integers(span, qlen))))
    a = np.array(rows, dtype=np.uint64).reshape(-1, 2)
    return O.oracle_sort128(a)


@pytest.mark.parametrize("seed", range(8))
def test_lchain_dp(seed):
    rng = np.random.default_rng(40 + seed)
    for it in range(25):
        a = make_anchors(rng, n_chain=int(rng.integers(1, 5)), n_noise=int(rng.integers(0, 400)))
        for (mdx, mdy, bw, skip, iters, mincnt, minsc, is_cdna) in [(5000, 5000, 500, 25, 5000, 3, 40, 0), (2000, 2000, 2000, 25, 50, 3, 100, 0), (200000, 2000, 200000, 25, 5000, 3, 40, 1)]:
            pg = np.float32(np.float32(0.8) * 0.01 * 15)
            x = O.oracle_lchain_dp(a, mdx, mdy, bw, skip, iters, mincnt, minsc, float(pg), 0.0, is_cdna)
            y = O.ref_lchain_dp(a, mdx, mdy, bw, skip, iters, mincnt, minsc, float(pg), 0.0, is_cdna)
            assert (x[0] == y[0]).all() and x[1].shape == y[1].shape and (x[1] == y[1]).all(), (it, mdx)


@pytest.mark.parametrize("seed", range(6))
def test_lchain_rmq(seed):
    """mg_lchain_rmq: the answer on equal priorities depends on the AVL shape of krmq.h -- checked against the reference
    over window sizes that force erasures, a tiny tree cap, with and without the inner tree"""
    rng = np.random.default_rng(900 + seed)
    for it in range(20):
        a = make_anchors(rng, n_chain=int(rng.integers(1, 5)), n_noise=int(rng.integers(0, 500)))
        for (md, mdi, bw, skip, cap, mincnt, minsc) in [(5000, 1000, 20000, 25, 100000, 3, 40), (800, 0, 500, 25, 100000, 3, 40),
                                                         (5000, 1000, 2000, 5, 12, 2, 20), (300, 300, 100, 25, 100000, 3, 40)]:
            pg = np.float32(np.float32(0.8) * 0.01 * 15)
            x = O.oracle_lchain_rmq(a, md, mdi, bw, skip, cap, mincnt, minsc, float(pg), 0.0)
            y = O.ref_lchain_rmq(a, md, mdi, bw, skip, cap, mincnt, minsc, float(pg), 0.0)
            assert len(x[0]) == len(y[0]) and (x[0] == y[0]).all() and x[1].shape == y[1].shape and (x[1] == y[1]).all(), (it, md, cap)


def _ref_extz2(q, t, mat, go, ge, w, zdrop, eb, flag):
    ez = O.RefEz()
    q = np.ascontiguousarray(q, dtype=np.uint8); t = np.ascontiguousarray(t, dtype=np.uint8); mat = np.ascontiguousarray(mat, dtype=np.int8)
    O.ref().refshim_extz2(C.c_int(len(q)), q.ctypes.data_as(C.c_void_p), C.c_int(len(t)), t.ctypes.data_as(C.c_void_p), C.c_int8(5),
                          mat.ctypes.data_as(C.c_void_p), C.c_int8(go), C.c_int8(ge), C.c_int(w), C.c_int(zdrop), C.c_int(eb), C.c_int(flag), C.byref(ez))
    d = O.ez_dict(ez, True)
    O.ref().refshim_free(ez.cigar)
    return d


def test_extz2_is_extd2_with_equal_gaps():
    """The single-affine kernel of the reference (ksw2_extz2_sse.c:26) is not rebuilt: for every flag combination align.c
    passes (KSW_EZ_APPROX_DROP is never set, align.c:336-368,779-890), it equals ksw_extd2 with q2 = q, e2 = e -- shown
    here on the reference itself and on the oracle, band-clipped calls included."""
    rng = np.random.default_rng(77)
    flags = [0, 0x08, 0x40, 0x40 | 0x02 | 0x80, 0x02, 0x40 | 0x02, 0x08 | 0x02, 0x01, 0x80]
    for it in range(1500):
        tl = int(rng.integers(1, 400)); t = rng.integers(0, 4, tl).astype(np.uint8)
        q = O.mutate(t, rng, err=float(rng.choice([0.0, 0.05, 0.15, 0.4])))
        if len(q) == 0:
            q = np.array([0], dtype=np.uint8)
        if rng.random() < 0.2:
            q[rng.integers(0, len(q))] = 4
        a, b, go, ge = [(2, 4, 4, 2), (1, 4, 6, 2), (2, 8, 12, 2), (1, 1, 1, 1), (2, 4, 24, 1)][it % 5]
        mat = O.simple_mat(a, b, 1)
        w = int(rng.choice([-1, 5, 17, 40, 100, 751])); zd = int(rng.choice([-1, 50, 200, 400])); eb = int(rng.choice([-1, 0, 10]))
        fl = int(rng.choice(flags))
        x = _ref_extz2(q, t, mat, go, ge, w, zd, eb, fl)
        assert x == O.ref_extd2(q, t, mat, go, ge, go, ge, w, zd, eb, fl), (it, fl)
        assert x == O.oracle_extd2(q, t, mat, go, ge, go, ge, w, zd, eb, fl), (it, fl)


def _spliced_pair(rng, n_exon, err):
    """target = exons separated by introns with (mostly) canonical GT..AG ends; query = the exons with errors"""
    ex = [rng.integers(0, 4, int(rng.integers(20, 120))).astype(np.uint8) for _ in range(n_exon)]
    t_parts = [ex[0]]
    for k in range(1, n_exon):
        il = int(rng.integers(30, 400))
        intron = rng.integers(0, 4, il).astype(np.uint8)
        sig = int(rng.integers(0, 5))
        if sig < 3: intron[:2] = [2, 3]; intron[-2:] = [0, 2]      # GT..AG
        elif sig == 3: intron[:2] = [2, 1]; intron[-2:] = [0, 2]    # GC..AG
        t_parts += [intron, ex[k]]
    t = np.concatenate(t_parts)
    q = O.mutate(np.concatenate(ex), rng, err=err)
    if len(q) == 0:
        q = np.array([0], dtype=np.uint8)
    return q, t


@pytest.mark.parametrize("seed", range(4))
def test_exts2_splice(seed):
    """ksw_exts2_sse (spliced alignment) restatement vs the reference: splice models, strands, reversed (left-extension)
    inputs, gap left/right alignment, extension mode, approximate max, annotated junctions and junction scores"""
    rng = np.random.default_rng(300 + seed)
    SPF, SPR, FLANK, CMPLX, SPSC = 0x100, 0x200, 0x400, 0x800, 0x1000
    base_flags = [0, 0x08, 0x40, 0x40 | 0x02 | 0x80, 0x02, 0x01, 0x80, 0x40 | 0x80]
    for it in range(220):
        q, t = _spliced_pair(rng, int(rng.integers(1, 5)), float(rng.choice([0.0, 0.03, 0.1])))
        if rng.random() < 0.15:
            q[rng.integers(0, len(q))] = 4
        if rng.random() < 0.3:  # reverse-complement both: the signals of the other transcript strand
            q = (3 - q[::-1]) % 4 if (q < 4).all() else q
            t = 3 - t[::-1]
        fl = int(rng.choice(base_flags)) | int(rng.choice([0, SPF, SPR])) | (FLANK if rng.random() < 0.5 else 0) | (CMPLX if rng.random() < 0.3 else 0)
        a, b, go, ge, go2, noncan = [(1, 2, 2, 1, 32, 9), (2, 4, 4, 2, 24, 5), (1, 2, 2, 1, 16, 0)][it % 3]
        mat = O.simple_mat(a, b, 1)
        zd = int(rng.choice([-1, 100, 200])); eb = int(rng.choice([-1, 0, 10]))
        junc = None; jb = 9; jp = 5
        if rng.random() < 0.4:
            junc = (rng.random(len(t)) < 0.03).astype(np.uint8) * rng.integers(1, 16, len(t)).astype(np.uint8)
            if rng.random() < 0.5:
                fl |= SPSC
                junc = np.where(rng.random(len(t)) < 0.05, rng.integers(0, 200, len(t)), 0xff).astype(np.uint8)
        x = O.oracle_exts2(q, t, mat, go, ge, go2, noncan, zd, eb, jb, jp, fl, junc)
        y = O.ref_exts2(q, t, mat, go, ge, go2, noncan, zd, eb, jb, jp, fl, junc)
        assert x == y, (it, hex(fl), len(q), len(t), {k: (x[k], y[k]) for k in x if x[k] != y[k] and k != "cigar"}, x["cigar"][:8], y["cigar"][:8])


def test_hit_tail_oracle_vs_reference():
    """mm_append_cigar + mm_fix_cigar + mm_update_extra (align.c:105-334): oracle/mm2o_extra.c against the reference's own static functions
    (oracle/_ref/libminimap2_refalign.so = the reference with align.c compiled into a unit that exports them)."""
    import os
    import tail_cases as T
    if not os.path.exists(T.REFALIGN_SO):
        pytest.skip("oracle/_ref/libminimap2_refalign.so not built")
    rng = np.random.default_rng(5)
    for i in range(3000):
        c = T.make_case(rng)
        assert T.same(T.run_oracle(c), T.run_reference(c)), i
    for q, e in ((6, 2), (5, 4), (16, 1)):
        for i in range(300):
            c = T.make_case(rng)
            assert T.same(T.run_oracle(c, q, e), T.run_reference(c, q, e)), (q, e, i)
