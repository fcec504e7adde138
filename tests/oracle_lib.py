"""ctypes access to the CHECKERS: oracle/libmm2oracle.so (our plain-C restatement) and
oracle/_ref/libminimap2_ref.so (the unmodified reference compiled by oracle/Makefile).
Test infrastructure only -- never imported by minimap2_b200/."""
import ctypes as C
import gzip
import hashlib
import json
import os
import subprocess
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "libmm2oracle.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libminimap2_ref.so")
REF_BIN = os.path.join(ORACLE_DIR, "_ref", "minimap2")


class M128(C.Structure):
    _fields_ = [("x", C.c_uint64), ("y", C.c_uint64)]


class OracleEz(C.Structure):  # mm2o_ez_t
    _fields_ = [("max", C.c_int32), ("zdropped", C.c_int32), ("max_q", C.c_int32), ("max_t", C.c_int32),
                ("mqe", C.c_int32), ("mqe_t", C.c_int32), ("mte", C.c_int32), ("mte_q", C.c_int32),
                ("score", C.c_int32), ("n_cigar", C.c_int32), ("reach_end", C.c_int32), ("m_cigar", C.c_int32),
                ("cigar", C.POINTER(C.c_uint32))]


class RefEz(C.Structure):  # ksw_extz_t (ksw2.h:34-43)
    _fields_ = [("max_zd", C.c_uint32), ("max_q", C.c_int), ("max_t", C.c_int), ("mqe", C.c_int), ("mqe_t", C.c_int),
                ("mte", C.c_int), ("mte_q", C.c_int), ("score", C.c_int), ("m_cigar", C.c_int), ("n_cigar", C.c_int),
                ("reach_end", C.c_int), ("cigar", C.POINTER(C.c_uint32))]


def build_oracle():
    if not os.path.exists(ORACLE_SO):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "oracle"], stdout=subprocess.DEVNULL)


_oracle = None
_ref = None


def oracle():
    global _oracle
    if _oracle is None:
        build_oracle()
        L = C.CDLL(ORACLE_SO)
        L.mm2o_sketch.restype = C.c_int
        L.mm2o_lchain_dp.restype = C.c_int
        if hasattr(L, 'mm2o_lchain_rmq'):
            L.mm2o_lchain_rmq.restype = C.c_int
        L.mm2o_ll_i16.restype = C.c_int
        _oracle = L
    return _oracle


def have_ref():
    return os.path.exists(REF_SO)


# ---------------- recorded reference results (tests/golden/ref/) ----------------
# Tests that compare with the unmodified reference read what it computed from recordings keyed by their inputs, so that they run
# (and never skip) where oracle/_ref cannot be built. MM2_RECORD_REF=1 runs the reference instead and rewrites the recording:
#   MM2_RECORD_REF=1 python -m pytest tests -m "gpu or gpu_ext or not gpu"      (where oracle/_ref is built; GPU-side asserts may fail)
RECORDED_DIR = os.path.join(ROOT, "tests", "golden", "ref")


def file_digest(path):
    with open(path, "rb") as f:
        data = f.read()
    if path.endswith(".gz"):
        data = gzip.decompress(data)  # the gzip header carries a time stamp
    return hashlib.sha256(data).hexdigest()


def line_digest(line):
    return hashlib.sha256(line.encode()).hexdigest()[:16]


def recorded(key, produce):
    """`produce()`'s JSON-able result, from the recording for `key` (a list of strings naming the inputs completely)"""
    path = os.path.join(RECORDED_DIR, hashlib.sha256("\0".join(key).encode()).hexdigest()[:20] + ".json")
    if os.environ.get("MM2_RECORD_REF") == "1":
        os.makedirs(RECORDED_DIR, exist_ok=True)
        with open(path, "w") as f:
            json.dump({"key": key, "result": produce()}, f, separators=(",", ":"))
            f.write("\n")
    assert os.path.exists(path), "no recorded reference result for %r: record it with MM2_RECORD_REF=1 where oracle/_ref is built" % (key,)
    with open(path) as f:
        rec = json.load(f)
    assert rec["key"] == key, (rec["key"], key)
    return rec["result"]


def cli_key(args, cwd=None):
    """`args` with every input file replaced by its name and content digest (temporary paths differ from run to run)"""
    key = []
    for a in args:
        p = os.path.join(cwd or "", a)
        key.append("%s@%s" % (os.path.basename(a), file_digest(p)[:16]) if os.path.isfile(p) else a)
    return key


def ref_cli_lines(args, cwd=None):
    """the reference CLI's stdout for `args` (no -t: the output does not depend on it) as line digests, SAM @PG dropped:
    dict(args=, cwd=, lines=) for assert_same_lines"""
    def produce():
        p = subprocess.run([REF_BIN, "-t", "4"] + args, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=1800)
        assert p.returncode == 0, p.stderr.decode()[-2000:]
        return [line_digest(l) for l in p.stdout.decode().splitlines() if not l.startswith("@PG")]
    return dict(args=args, cwd=cwd, lines=recorded(["minimap2"] + cli_key(args, cwd), produce))


def assert_same_lines(got, ref):
    """`got` (output lines, SAM @PG dropped here) equals the reference output `ref` of ref_cli_lines, line by line"""
    got = [l for l in got if not l.startswith("@PG")]
    how = ("only digests of the reference's lines are stored; where oracle/_ref is built, `%s` (in %s) prints them"
           % (" ".join([REF_BIN] + ref["args"]), ref["cwd"] or os.getcwd()))
    assert len(got) == len(ref["lines"]), "%d output lines, the reference has %d (%s)" % (len(got), len(ref["lines"]), how)
    for i, (l, d) in enumerate(zip(got, ref["lines"])):
        assert line_digest(l) == d, "line %d differs from the reference's (%s):\ngot: %s" % (i, how, l[:600])
    return len(got)


def ref():
    global _ref
    if _ref is None:
        L = C.CDLL(REF_SO)
        L.refshim_sketch.restype = C.c_int
        L.refshim_lchain_dp.restype = C.c_int
        L.refshim_lchain_rmq.restype = C.c_int
        L.refshim_ll_i16.restype = C.c_int
        _ref = L
    return _ref


def ez_dict(ez, is_ref):
    if is_ref:
        mx, zd = ez.max_zd & 0x7fffffff, ez.max_zd >> 31
    else:
        mx, zd = ez.max, ez.zdropped
    cig = [ez.cigar[i] for i in range(ez.n_cigar)]
    return dict(max=mx, zdropped=zd, max_q=ez.max_q, max_t=ez.max_t, mqe=ez.mqe, mqe_t=ez.mqe_t, mte=ez.mte,
                mte_q=ez.mte_q, score=ez.score, n_cigar=ez.n_cigar, reach_end=ez.reach_end, cigar=cig)


def simple_mat(a, b, sc_ambi, transition=0):
    """align.c:11-38 ksw_gen_simple_mat / ksw_gen_ts_mat for m=5"""
    m = 5
    a = abs(a); b = -abs(b); sa = -abs(sc_ambi)
    mat = np.zeros(25, dtype=np.int8)
    for i in range(m - 1):
        for j in range(m - 1):
            mat[i * m + j] = a if i == j else b
        mat[i * m + m - 1] = sa
    for j in range(m):
        mat[(m - 1) * m + j] = sa
    if transition != 0 and -abs(transition) != b:
        t = -abs(transition)
        mat[0 * m + 2] = t; mat[1 * m + 3] = t; mat[2 * m + 0] = t; mat[3 * m + 1] = t
    return mat


def oracle_extd2(q, t, mat, gapo, gape, gapo2, gape2, w, zdrop, end_bonus, flag, m=5):
    ez = OracleEz()
    q = np.ascontiguousarray(q, dtype=np.uint8); t = np.ascontiguousarray(t, dtype=np.uint8)
    mat = np.ascontiguousarray(mat, dtype=np.int8)
    oracle().mm2o_extd2(C.c_int(len(q)), q.ctypes.data_as(C.c_void_p), C.c_int(len(t)), t.ctypes.data_as(C.c_void_p), C.c_int(m),
                        mat.ctypes.data_as(C.c_void_p), C.c_int(gapo), C.c_int(gape), C.c_int(gapo2), C.c_int(gape2),
                        C.c_int(w), C.c_int(zdrop), C.c_int(end_bonus), C.c_int(flag), C.byref(ez))
    d = ez_dict(ez, False)
    oracle().mm2o_free(ez.cigar)
    return d


def ref_extd2(q, t, mat, gapo, gape, gapo2, gape2, w, zdrop, end_bonus, flag, m=5):
    ez = RefEz()
    q = np.ascontiguousarray(q, dtype=np.uint8); t = np.ascontiguousarray(t, dtype=np.uint8)
    mat = np.ascontiguousarray(mat, dtype=np.int8)
    ref().refshim_extd2(C.c_int(len(q)), q.ctypes.data_as(C.c_void_p), C.c_int(len(t)), t.ctypes.data_as(C.c_void_p), C.c_int8(m),
                        mat.ctypes.data_as(C.c_void_p), C.c_int8(gapo), C.c_int8(gape), C.c_int8(gapo2), C.c_int8(gape2),
                        C.c_int(w), C.c_int(zdrop), C.c_int(end_bonus), C.c_int(flag), C.byref(ez))
    d = ez_dict(ez, True)
    ref().refshim_free(ez.cigar)
    return d


def _m128_array(a):
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 2)
    return a


def oracle_sketch(seq: bytes, w, k, rid=0, is_hpc=0):
    out = np.zeros((max(len(seq), 1), 2), dtype=np.uint64)
    n = oracle().mm2o_sketch(C.c_char_p(seq), C.c_int(len(seq)), C.c_int(w), C.c_int(k), C.c_uint32(rid), C.c_int(is_hpc),
                             out.ctypes.data_as(C.c_void_p))
    return out[:n].copy()


def ref_sketch(seq: bytes, w, k, rid=0, is_hpc=0):
    p = C.POINTER(M128)()
    n = ref().refshim_sketch(C.c_char_p(seq), C.c_int(len(seq)), C.c_int(w), C.c_int(k), C.c_uint32(rid), C.c_int(is_hpc), C.byref(p))
    out = np.zeros((n, 2), dtype=np.uint64)
    if n:
        C.memmove(out.ctypes.data, p, n * 16)
    ref().refshim_free(p)
    return out


def _chain_call(fn, args, a):
    a = _m128_array(a)
    u = C.POINTER(C.c_uint64)(); b = C.POINTER(M128)(); n_a = C.c_int(0)
    n_u = fn(*args, C.c_int64(len(a)), a.ctypes.data_as(C.c_void_p), C.byref(u), C.byref(b), C.byref(n_a))
    uu = np.array([u[i] for i in range(n_u)], dtype=np.uint64)
    bb = np.zeros((n_a.value, 2), dtype=np.uint64)
    if n_a.value:
        C.memmove(bb.ctypes.data, b, n_a.value * 16)
    return uu, bb, u, b


def oracle_lchain_dp(a, max_dist_x, max_dist_y, bw, max_skip, max_iter, min_cnt, min_sc, pen_gap, pen_skip, is_cdna=0, n_seg=1):
    args = [C.c_int(max_dist_x), C.c_int(max_dist_y), C.c_int(bw), C.c_int(max_skip), C.c_int(max_iter), C.c_int(min_cnt),
            C.c_int(min_sc), C.c_float(pen_gap), C.c_float(pen_skip), C.c_int(is_cdna), C.c_int(n_seg)]
    uu, bb, u, b = _chain_call(oracle().mm2o_lchain_dp, args, a)
    oracle().mm2o_free(u); oracle().mm2o_free(b)
    return uu, bb


def ref_lchain_dp(a, max_dist_x, max_dist_y, bw, max_skip, max_iter, min_cnt, min_sc, pen_gap, pen_skip, is_cdna=0, n_seg=1):
    args = [C.c_int(max_dist_x), C.c_int(max_dist_y), C.c_int(bw), C.c_int(max_skip), C.c_int(max_iter), C.c_int(min_cnt),
            C.c_int(min_sc), C.c_float(pen_gap), C.c_float(pen_skip), C.c_int(is_cdna), C.c_int(n_seg)]
    uu, bb, u, b = _chain_call(ref().refshim_lchain_dp, args, a)
    ref().refshim_free(u); ref().refshim_free(b)
    return uu, bb


def oracle_lchain_rmq(a, max_dist, max_dist_inner, bw, max_skip, cap, min_cnt, min_sc, pen_gap, pen_skip):
    args = [C.c_int(max_dist), C.c_int(max_dist_inner), C.c_int(bw), C.c_int(max_skip), C.c_int(cap), C.c_int(min_cnt),
            C.c_int(min_sc), C.c_float(pen_gap), C.c_float(pen_skip)]
    uu, bb, u, b = _chain_call(oracle().mm2o_lchain_rmq, args, a)
    oracle().mm2o_free(u); oracle().mm2o_free(b)
    return uu, bb


def ref_lchain_rmq(a, max_dist, max_dist_inner, bw, max_skip, cap, min_cnt, min_sc, pen_gap, pen_skip):
    args = [C.c_int(max_dist), C.c_int(max_dist_inner), C.c_int(bw), C.c_int(max_skip), C.c_int(cap), C.c_int(min_cnt),
            C.c_int(min_sc), C.c_float(pen_gap), C.c_float(pen_skip)]
    uu, bb, u, b = _chain_call(ref().refshim_lchain_rmq, args, a)
    ref().refshim_free(u); ref().refshim_free(b)
    return uu, bb


def oracle_sort128(a):
    a = _m128_array(a).copy()
    oracle().mm2o_radix_sort_128x(a.ctypes.data_as(C.c_void_p), C.c_void_p(a.ctypes.data + a.nbytes))
    return a


def ref_sort128(a):
    a = _m128_array(a).copy()
    ref().refshim_sort128x(a.ctypes.data_as(C.c_void_p), C.c_int64(len(a)))
    return a


def oracle_ll_i16(q, t, mat, gapo, gape, m=5):
    q = np.ascontiguousarray(q, dtype=np.uint8); t = np.ascontiguousarray(t, dtype=np.uint8)
    mat = np.ascontiguousarray(mat, dtype=np.int8)
    qe = C.c_int(); te = C.c_int()
    sc = oracle().mm2o_ll_i16(C.c_int(len(q)), q.ctypes.data_as(C.c_void_p), C.c_int(len(t)), t.ctypes.data_as(C.c_void_p), C.c_int(m),
                              mat.ctypes.data_as(C.c_void_p), C.c_int(gapo), C.c_int(gape), C.byref(qe), C.byref(te))
    return sc, qe.value, te.value


def ref_ll_i16(q, t, mat, gapo, gape, m=5):
    q = np.ascontiguousarray(q, dtype=np.uint8); t = np.ascontiguousarray(t, dtype=np.uint8)
    mat = np.ascontiguousarray(mat, dtype=np.int8)
    qe = C.c_int(); te = C.c_int()
    sc = ref().refshim_ll_i16(C.c_int(len(q)), q.ctypes.data_as(C.c_void_p), C.c_int(len(t)), t.ctypes.data_as(C.c_void_p), C.c_int(m),
                              mat.ctypes.data_as(C.c_void_p), C.c_int(gapo), C.c_int(gape), C.byref(qe), C.byref(te))
    return sc, qe.value, te.value


# ---------------- synthetic data helpers shared by tests and bench ----------------
def mutate(seq: np.ndarray, rng, err=0.1, sub=0.4, ins=0.25, dele=0.35):
    """ONT-like error profile on an nt4 array (SURVEY 8d): err split sub/ins/del."""
    out = []
    r = rng.random(len(seq))
    kind = rng.random(len(seq))
    newb = rng.integers(0, 4, len(seq))
    for i in range(len(seq)):
        if r[i] < err:
            if kind[i] < sub:
                out.append((int(seq[i]) + 1 + int(newb[i]) % 3) % 4)
            elif kind[i] < sub + ins:
                out.append(int(seq[i])); out.append(int(newb[i]))
            else:
                pass
        else:
            out.append(int(seq[i]))
    return np.array(out, dtype=np.uint8)


# ---------------- ksw_exts2 (splice): oracle restatement and reference ----------------
def _exts2_args(q, t, mat, gapo, gape, gapo2, noncan, zdrop, end_bonus, junc_bonus, junc_pen, flag, junc, i8):
    q = np.ascontiguousarray(q, dtype=np.uint8); t = np.ascontiguousarray(t, dtype=np.uint8)
    mat = np.ascontiguousarray(mat, dtype=np.int8)
    T = C.c_int8 if i8 else C.c_int
    jp = None if junc is None else np.ascontiguousarray(junc, dtype=np.uint8)
    args = [C.c_int(len(q)), q.ctypes.data_as(C.c_void_p), C.c_int(len(t)), t.ctypes.data_as(C.c_void_p), T(5), mat.ctypes.data_as(C.c_void_p),
            T(gapo), T(gape), T(gapo2), T(noncan), C.c_int(zdrop), C.c_int(end_bonus), T(junc_bonus), T(junc_pen), C.c_int(flag),
            C.c_void_p(0) if jp is None else jp.ctypes.data_as(C.c_void_p)]
    return args, (q, t, mat, jp)


def oracle_exts2(q, t, mat, gapo, gape, gapo2, noncan, zdrop, end_bonus, junc_bonus, junc_pen, flag, junc=None):
    ez = OracleEz()
    args, keep = _exts2_args(q, t, mat, gapo, gape, gapo2, noncan, zdrop, end_bonus, junc_bonus, junc_pen, flag, junc, False)
    oracle().mm2o_exts2(*args, C.byref(ez))
    d = ez_dict(ez, False)
    oracle().mm2o_free(ez.cigar)
    return d


def ref_exts2(q, t, mat, gapo, gape, gapo2, noncan, zdrop, end_bonus, junc_bonus, junc_pen, flag, junc=None):
    ez = RefEz()
    args, keep = _exts2_args(q, t, mat, gapo, gape, gapo2, noncan, zdrop, end_bonus, junc_bonus, junc_pen, flag, junc, True)
    ref().refshim_exts2(*args, C.byref(ez))
    d = ez_dict(ez, True)
    ref().refshim_free(ez.cigar)
    return d


# ---------------- seeding stage (oracle index + anchors) ----------------
class OracleIndex:
    def __init__(self, seqs, names, w, k, is_hpc=0):
        L = oracle()
        L.mm2o_idx_build.restype = C.c_void_p
        n = len(seqs)
        self._seqs = [s if isinstance(s, bytes) else bytes(s) for s in seqs]
        arr = (C.c_char_p * n)(*self._seqs)
        lens = (C.c_int * n)(*[len(s) for s in self._seqs])
        nm = (C.c_char_p * n)(*[x.encode() for x in names])
        self.names = list(names)
        self.h = C.c_void_p(L.mm2o_idx_build(n, arr, lens, nm, w, k, is_hpc))

    def anchors(self, seq, qname=None, flag=0, mid_occ=10, q_occ_frac=0.01, max_max_occ=4095, occ_dist=500):
        L = oracle()
        L.mm2o_collect_seed_hits.restype = C.c_int64
        a = C.POINTER(M128)(); mp = C.POINTER(C.c_uint64)(); rep = C.c_int(0); nmp = C.c_int(0)
        s = seq if isinstance(seq, bytes) else bytes(seq)
        n = L.mm2o_collect_seed_hits(self.h, None if qname is None else qname.encode(), s, C.c_int(len(s)), C.c_int64(flag), C.c_int(mid_occ),
                                     C.c_float(q_occ_frac), C.c_int(max_max_occ), C.c_int(occ_dist), C.byref(a), C.byref(rep), C.byref(nmp), C.byref(mp))
        out = np.zeros((n, 2), dtype=np.uint64)
        if n:
            C.memmove(out.ctypes.data, a, n * 16)
        mini = np.array([mp[i] for i in range(nmp.value)], dtype=np.uint64)
        L.mm2o_free(a); L.mm2o_free(mp)
        return out, rep.value, mini

    def close(self):
        if self.h:
            oracle().mm2o_idx_destroy(self.h)
            self.h = None
