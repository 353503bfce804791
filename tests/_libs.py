"""ctypes bindings used by the tests: the compiled reference (oracle/_ref/libmm2ref.so,
when present), the plain-C oracle port (oracle/_ref/libmm2oracle.so) and helpers.
Test infrastructure only."""
import ctypes as C
import hashlib
import json
import os
import subprocess
import tempfile
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libmm2ref.so")
ORC_SO = os.path.join(ORACLE_DIR, "_ref", "libmm2oracle.so")
REF_BIN_A = os.path.join(ORACLE_DIR, "_ref", "minimap2_A")
REF_BIN_B = os.path.join(ORACLE_DIR, "_ref", "minimap2_B")

mm128 = np.dtype([("x", "<u8"), ("y", "<u8")])


class Extz(C.Structure):  # orc_extz_t
    _fields_ = [("max", C.c_uint32), ("zdropped", C.c_int), ("max_q", C.c_int), ("max_t", C.c_int),
                ("mqe", C.c_int), ("mqe_t", C.c_int), ("mte", C.c_int), ("mte_q", C.c_int), ("score", C.c_int),
                ("m_cigar", C.c_int), ("n_cigar", C.c_int), ("reach_end", C.c_int), ("cigar", C.POINTER(C.c_uint32))]


class RefExtz(C.Structure):  # ksw_extz_t (ksw2.h:23-32)
    _fields_ = [("max_zd", C.c_uint32), ("max_q", C.c_int), ("max_t", C.c_int), ("mqe", C.c_int), ("mqe_t", C.c_int),
                ("mte", C.c_int), ("mte_q", C.c_int), ("score", C.c_int), ("m_cigar", C.c_int), ("n_cigar", C.c_int),
                ("reach_end", C.c_int), ("cigar", C.POINTER(C.c_uint32))]


def build_oracle():
    if not os.path.exists(ORC_SO) or os.path.getmtime(ORC_SO) < os.path.getmtime(os.path.join(ORACLE_DIR, "mm2_oracle.c")):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "port"], stdout=subprocess.DEVNULL)


_orc = None
_ref = None
libc = C.CDLL("libc.so.6")
libc.malloc.restype = C.c_void_p
libc.free.argtypes = [C.c_void_p]


def oracle():
    global _orc
    if _orc is None:
        build_oracle()
        L = C.CDLL(ORC_SO)
        L.orc_sketch.restype = C.c_int
        L.orc_sketch.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_int, C.c_void_p, C.c_int]
        L.orc_idx_build.restype = C.c_void_p
        L.orc_idx_build.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_char_p)]
        L.orc_idx_destroy.argtypes = [C.c_void_p]
        L.orc_idx_get.restype = C.POINTER(C.c_uint64)
        L.orc_idx_get.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_int)]
        L.orc_idx_cal_max_occ.restype = C.c_int32
        L.orc_idx_cal_max_occ.argtypes = [C.c_void_p, C.c_float]
        L.orc_idx_n_minimizers.restype = C.c_int64
        L.orc_idx_n_minimizers.argtypes = [C.c_void_p]
        L.orc_collect_seeds.restype = C.c_int64
        L.orc_collect_seeds.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                        C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p]
        L.orc_chain_dp.restype = C.c_int
        L.orc_chain_dp.argtypes = [C.c_int] * 9 + [C.c_int64, C.c_void_p, C.c_void_p]
        L.orc_ksw_extd2.restype = None
        L.orc_ksw_extd2.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int8, C.c_void_p, C.c_int8, C.c_int8,
                                    C.c_int8, C.c_int8, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(Extz)]
        L.orc_ksw_band_cells.restype = C.c_int64
        L.orc_ksw_band_cells.argtypes = [C.c_int, C.c_int, C.c_int]
        L.orc_radix_sort_128x.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_radix_sort_64.argtypes = [C.c_void_p, C.c_void_p]
        _orc = L
    return _orc


def have_ref():
    return os.path.exists(REF_SO)


def have_ref_bin():
    return os.path.exists(REF_BIN_B)


DIGESTS = os.path.join(ROOT, "tests", "golden", "digests.json")


def _bytes(out):
    if isinstance(out, (list, tuple)):
        return b"\n".join(l if isinstance(l, bytes) else l.encode() for l in out)
    return out


def check_digest(key, out):
    """Where the reference fork (oracle/_ref) is not built, an output that the tests compare with the reference's is compared
    with the size and sha256 kept for key in tests/golden/digests.json; each entry's "source" says whose output it is.
    out: bytes, or a list of lines (str or bytes).  On a mismatch the output is saved to a temporary file for a line-by-line
    diff against a run of the reference elsewhere."""
    with open(DIGESTS) as f:
        want = json.load(f).get(key)
    assert want is not None, f"no recorded digest for {key!r} in {DIGESTS}"
    b = _bytes(out)
    got = {"bytes": len(b), "sha256": hashlib.sha256(b).hexdigest()}
    if got != {k: want[k] for k in got}:
        fd, path = tempfile.mkstemp(prefix="airlift_digest_", suffix=".out")
        with os.fdopen(fd, "wb") as f:
            f.write(b)
        raise AssertionError(f"{key}: output {got} differs from the recorded one {want}; output saved to {path}")


def record_reference_digest(key, want):
    """With AIRLIFT_RECORD_REFERENCE_DIGESTS=1, stores the digest of want -- the REFERENCE's output, already compared with this
    project's by the caller -- as the entry of key in tests/golden/digests.json.  Only the reference branches of the tests call it."""
    if os.environ.get("AIRLIFT_RECORD_REFERENCE_DIGESTS") != "1":
        return
    b = _bytes(want)
    with open(DIGESTS) as f:
        d = json.load(f)
    d[key] = {"bytes": len(b), "sha256": hashlib.sha256(b).hexdigest(), "source": "reference fork (oracle/_ref)"}
    with open(DIGESTS, "w") as f:
        json.dump(d, f, indent=1, sort_keys=True)


class mm128_v(C.Structure):
    _fields_ = [("n", C.c_size_t), ("m", C.c_size_t), ("a", C.c_void_p)]


def ref():
    global _ref
    if _ref is None:
        L = C.CDLL(REF_SO)
        L.mm_sketch.restype = None
        L.mm_sketch.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_int, C.POINTER(mm128_v)]
        L.mm_idx_str.restype = C.c_void_p
        L.mm_idx_str.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p)]
        L.mm_idx_destroy.argtypes = [C.c_void_p]
        L.mm_idx_get.restype = C.POINTER(C.c_uint64)
        L.mm_idx_get.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_int)]
        L.mm_idx_cal_max_occ.restype = C.c_int32
        L.mm_idx_cal_max_occ.argtypes = [C.c_void_p, C.c_float]
        L.ref_collect_seeds.restype = C.c_void_p
        L.ref_collect_seeds.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                        C.POINTER(C.c_int64), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_void_p)]
        L.ref_chain_dp.restype = C.c_int
        L.ref_chain_dp.argtypes = [C.c_int] * 9 + [C.c_int64, C.c_void_p, C.c_void_p]
        L.ksw_extd2_sse.restype = None
        L.ksw_extd2_sse.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int8, C.c_void_p, C.c_int8,
                                    C.c_int8, C.c_int8, C.c_int8, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(RefExtz)]
        L.radix_sort_128x.argtypes = [C.c_void_p, C.c_void_p]
        L.radix_sort_64.argtypes = [C.c_void_p, C.c_void_p]
        _ref = L
    return _ref


# ----------------------------------------------------------------- wrappers

def orc_sketch(seq: bytes, w, k, rid=0, hpc=0):
    out = np.zeros(len(seq) + 1, dtype=mm128)
    n = oracle().orc_sketch(seq, len(seq), w, k, rid, hpc, out.ctypes.data, len(out))
    return out[:n].copy()


def ref_sketch(seq: bytes, w, k, rid=0, hpc=0):
    v = mm128_v(0, 0, None)
    ref().mm_sketch(None, seq, len(seq), w, k, rid, hpc, C.byref(v))
    out = np.zeros(v.n, dtype=mm128)
    if v.n:
        C.memmove(out.ctypes.data, v.a, v.n * 16)
    libc.free(v.a)
    return out


def frag_minimizers(sketch_fn, segs, w, k):
    """collect_minimizers (map.c:64-77): rid = segment index, y += (sum of previous lengths)<<1."""
    parts, tot = [], 0
    for i, s in enumerate(segs):
        a = sketch_fn(s, w, k, i)
        a["y"] += np.uint64(tot << 1)
        parts.append(a)
        tot += len(s)
    return (np.concatenate(parts) if parts else np.zeros(0, dtype=mm128)), tot


def c_str_array(seqs):
    arr = (C.c_char_p * len(seqs))()
    for i, s in enumerate(seqs):
        arr[i] = s
    return arr


def orc_collect(idx, heap, flag, max_occ, mv, qlen):
    L = oracle()
    rep = C.c_int(0)
    nmp = C.c_int(0)
    mv = np.ascontiguousarray(mv)
    n_a = L.orc_collect_seeds(idx, heap, flag, max_occ, len(mv), mv.ctypes.data, qlen, None, C.byref(rep), C.byref(nmp), None)
    a = np.zeros(n_a + 1, dtype=mm128)
    mp = np.zeros(len(mv) + 1, dtype=np.uint64)
    n_a = L.orc_collect_seeds(idx, heap, flag, max_occ, len(mv), mv.ctypes.data, qlen, a.ctypes.data, C.byref(rep), C.byref(nmp), mp.ctypes.data)
    return a[:n_a].copy(), rep.value, mp[:nmp.value].copy()


def ref_collect(mi, heap, flag, max_occ, mv, qlen):
    L = ref()
    n_a = C.c_int64(0)
    rep = C.c_int(0)
    nmp = C.c_int(0)
    mpp = C.c_void_p(0)
    mv = np.ascontiguousarray(mv)
    p = L.ref_collect_seeds(mi, heap, flag, max_occ, len(mv), mv.ctypes.data, qlen, C.byref(n_a), C.byref(rep), C.byref(nmp), C.byref(mpp))
    a = np.zeros(n_a.value, dtype=mm128)
    if n_a.value:
        C.memmove(a.ctypes.data, p, n_a.value * 16)
    mp = np.zeros(nmp.value, dtype=np.uint64)
    if nmp.value:
        C.memmove(mp.ctypes.data, mpp.value, nmp.value * 8)
    libc.free(p)
    libc.free(mpp)
    return a, rep.value, mp


def chain_call(fn, params, a):
    """params = (max_dist_x, max_dist_y, bw, max_skip, max_iter, min_cnt, min_sc, is_cdna, n_segs)"""
    a = np.ascontiguousarray(a.copy())
    u = np.zeros(len(a) + 1, dtype=np.uint64)
    n_u = fn(*params, len(a), a.ctypes.data, u.ctypes.data)
    u = u[:n_u].copy()
    n_v = int((u & np.uint64(0xffffffff)).sum())
    return u, a[:n_v].copy()


def _extz_tuple(ez, zd, mx):
    cig = [ez.cigar[i] for i in range(ez.n_cigar)]
    return dict(max=mx, zdropped=zd, max_q=ez.max_q, max_t=ez.max_t, mqe=ez.mqe, mqe_t=ez.mqe_t, mte=ez.mte,
                mte_q=ez.mte_q, score=ez.score, reach_end=ez.reach_end, cigar=cig)


def simple_mat(a, b, sc_ambi):
    """ksw_gen_simple_mat (align.c:9-22) for m=5."""
    m = np.zeros(25, dtype=np.int8)
    a, b, sc_ambi = abs(a), -abs(b), -abs(sc_ambi)
    for i in range(4):
        for j in range(4):
            m[i * 5 + j] = a if i == j else b
        m[i * 5 + 4] = sc_ambi
    for j in range(5):
        m[20 + j] = sc_ambi
    return m


class KswScoring:
    """One scoring of the DP kernels with the job parameters the tests use with it.  b and sc_ambi may be given with either sign:
    simple_mat, like make_score on the device and ksw_gen_simple_mat in the reference, takes their magnitude."""

    def __init__(self, name, a, b, sc_ambi, q, e, q2, e2, zdrop, end_bonus, band):
        self.name, self.a, self.b, self.sc_ambi = name, a, b, sc_ambi
        self.q, self.e, self.q2, self.e2 = q, e, q2, e2
        self.zdrop, self.end_bonus, self.band = zdrop, end_bonus, band

    @property
    def mat(self):
        return simple_mat(self.a, self.b, self.sc_ambi)

    @property
    def pen(self):
        return (self.q, self.e, self.q2, self.e2)

    def set_opt(self, opt):
        """the scoring fields of an api.MapOpt, as the CLI or mappy would set them"""
        opt.a, opt.b, opt.q, opt.e, opt.q2, opt.e2, opt.sc_ambi = self.a, self.b, self.q, self.e, self.q2, self.e2, self.sc_ambi
        return opt

    def __repr__(self):
        return self.name


# Every scoring the DP kernels are held to the oracle under.  sr and ont are the presets' own; the asm presets (host/opts.c) come
# close to the int8 limit of the reference's lanes, (q+e)+(q2+e2) <= 127, and edge127 sits on it; eq is the single-affine case
# (q == q2, e == e2); N0 gives N a zero score, which ksw2 replaces by -e2; bigA has large scores and a large N penalty; under
# bail the worst score exceeds 2(q+e), where ksw2 returns before any DP.  asm20 gives b negative, bigA sc_ambi negative.
KSW_SCORINGS = {s.name: s for s in [
    KswScoring("sr", 2, 8, 1, 12, 2, 24, 1, 100, 10, 151),
    KswScoring("ont", 2, 4, 1, 4, 2, 24, 1, 400, -1, 751),          # map-ont
    KswScoring("asm5", 1, 19, 1, 39, 3, 81, 1, 200, -1, 500),
    KswScoring("asm10", 1, 9, 1, 16, 2, 41, 1, 200, 5, 500),
    KswScoring("asm20", 1, -4, 1, 6, 2, 26, 1, 200, 10, 500),
    KswScoring("edge127", 1, 20, 1, 40, 3, 83, 1, 400, 10, 500),
    KswScoring("eq", 1, 4, 1, 6, 1, 6, 1, 200, 5, 200),
    KswScoring("N0", 2, 4, 0, 4, 2, 24, 1, 400, -1, 751),
    KswScoring("bigA", 10, 20, -5, 20, 4, 60, 2, 300, 20, 300),
    KswScoring("bail", 2, 20, 1, 4, 2, 24, 1, 100, 10, 151),
]}


def orc_ksw(q, t, mat, gq, ge, gq2, ge2, w, zdrop, end_bonus, flag):
    ez = Extz()
    q = np.ascontiguousarray(q, dtype=np.uint8)
    t = np.ascontiguousarray(t, dtype=np.uint8)
    oracle().orc_ksw_extd2(len(q), q.ctypes.data, len(t), t.ctypes.data, 5, mat.ctypes.data, gq, ge, gq2, ge2, w, zdrop, end_bonus, flag, C.byref(ez))
    r = _extz_tuple(ez, ez.zdropped, ez.max)
    libc.free(ez.cigar)
    return r


def ref_ksw(q, t, mat, gq, ge, gq2, ge2, w, zdrop, end_bonus, flag):
    ez = RefExtz()
    C.memset(C.byref(ez), 0, C.sizeof(ez))
    q = np.ascontiguousarray(q, dtype=np.uint8)
    t = np.ascontiguousarray(t, dtype=np.uint8)
    ref().ksw_extd2_sse(None, len(q), q.ctypes.data, len(t), t.ctypes.data, 5, mat.ctypes.data, gq, ge, gq2, ge2, w, zdrop, end_bonus, flag, C.byref(ez))
    r = _extz_tuple(ez, ez.max_zd >> 31, ez.max_zd & 0x7fffffff)
    libc.free(ez.cigar)
    return r


# ----------------------------------------------------------------- data

def rand_seq(rng, n, n_frac=0.0):
    s = rng.integers(0, 4, n)
    b = np.frombuffer(b"ACGT", dtype=np.uint8)[s].copy()
    if n_frac > 0:
        b[rng.random(n) < n_frac] = ord("N")
    return b.tobytes()


def mutate(rng, s: bytes, sub=0.01, ins=0.002, dele=0.002):
    out = bytearray()
    for ch in s:
        u = rng.random()
        if u < dele:
            continue
        if u < dele + ins:
            out.append(b"ACGT"[rng.integers(0, 4)])
        if u < dele + ins + sub:
            out.append(b"ACGT"[rng.integers(0, 4)])
        else:
            out.append(ch)
    return bytes(out)


_COMP = bytes.maketrans(b"ACGTacgt", b"TGCAtgca")


def revcomp(s: bytes):
    return s.translate(_COMP)[::-1]


def nt4(s: bytes):
    t = np.full(256, 4, dtype=np.uint8)
    for i, ch in enumerate(b"ACGT"):
        t[ch] = i
        t[ch + 32] = i
    t[ord("U")] = t[ord("u")] = 3
    return t[np.frombuffer(s, dtype=np.uint8)]
