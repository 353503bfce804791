"""mappy-compatible Python interface to the B200 mapper (libmm2b200.so through ctypes).

    from airlift_b200 import mappy as mp
    a = mp.Aligner("ref.fa", preset="map-ont")
    for hit in a.map(seq):
        print(hit)

Aligner, Alignment, ThreadBuffer, fastx_read, revcomp and verbose behave as the reference's mappy 2.17 does.  Mapping runs on
the GPU: map() goes through mm_map_frag, whose calls from any number of threads are mapped together as shared mini-batches on
every GPU of the index; ctypes releases the GIL for each foreign call, so Python threads reach that queue at the same time.
Aligner.map_batch() maps a list of reads as whole mini-batches, the throughput path.

What differs from the reference's mappy:
  - options this build does not implement (splice presets, MM_F_SPLICE in extra_flags, ...) raise ValueError with the
    library's message, and a missing CUDA device raises RuntimeError, both before anything is read;
  - a failure inside a mapping round still ends the process, as it does for C callers of mm_map_frag;
  - the hits of read 2 of a pair are reported in read 2's own orientation (strand and query coordinates), as the PAF writer
    prints a pair;
  - map() and map_batch() take an optional read name: it seeds the choice among equally good chains, as the read names of
    a FASTQ file do on the command line.
"""
import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmm2b200.so")

MM_F_CIGAR = 0x004
MM_F_SPLICE = 0x080
MM_F_INDEPEND_SEG = 0x20000
MM_I_HPC = 0x1
MM_B200_HITS_COLS = 22
MM_B200_HITS_CS, MM_B200_HITS_MD = 0x1, 0x2
(_FRAG, _SEG, _RID, _RS, _RE, _QS, _QE, _REV, _MAPQ, _PRI, _MLEN, _BLEN, _N_AMBI, _TS, _DP_SCORE, _DP_MAX, _N_CIGAR, _CIGAR_OFF,
 _CS_OFF, _CS_LEN, _MD_OFF, _MD_LEN) = range(MM_B200_HITS_COLS)


class IdxOpt(C.Structure):  # mm_idxopt_t
    _fields_ = [("k", C.c_short), ("w", C.c_short), ("flag", C.c_short), ("bucket_bits", C.c_short), ("mini_batch_size", C.c_int),
                ("batch_size", C.c_uint64)]


class MapOpt(C.Structure):  # mm_mapopt_t (include/minimap_b200.h)
    _fields_ = [("flag", C.c_int64), ("seed", C.c_int), ("sdust_thres", C.c_int), ("max_qlen", C.c_int), ("bw", C.c_int),
                ("max_gap", C.c_int), ("max_gap_ref", C.c_int), ("max_frag_len", C.c_int), ("max_chain_skip", C.c_int),
                ("max_chain_iter", C.c_int), ("min_cnt", C.c_int), ("min_chain_score", C.c_int), ("mask_level", C.c_float),
                ("pri_ratio", C.c_float), ("best_n", C.c_int), ("max_join_long", C.c_int), ("max_join_short", C.c_int),
                ("min_join_flank_sc", C.c_int), ("min_join_flank_ratio", C.c_float), ("a", C.c_int), ("b", C.c_int), ("q", C.c_int),
                ("e", C.c_int), ("q2", C.c_int), ("e2", C.c_int), ("sc_ambi", C.c_int), ("noncan", C.c_int), ("junc_bonus", C.c_int),
                ("zdrop", C.c_int), ("zdrop_inv", C.c_int), ("end_bonus", C.c_int), ("min_dp_max", C.c_int), ("min_ksw_len", C.c_int),
                ("anchor_ext_len", C.c_int), ("anchor_ext_shift", C.c_int), ("max_clip_ratio", C.c_float), ("pe_ori", C.c_int),
                ("pe_bonus", C.c_int), ("mid_occ_frac", C.c_float), ("min_mid_occ", C.c_int32), ("mid_occ", C.c_int32),
                ("max_occ", C.c_int32), ("mini_batch_size", C.c_int), ("max_sw_mat", C.c_int64), ("split_prefix", C.c_char_p)]


class _IdxHead(C.Structure):  # leading fields of mm_idx_t
    _fields_ = [("b", C.c_int32), ("w", C.c_int32), ("k", C.c_int32), ("flag", C.c_int32), ("n_seq", C.c_uint32)]


class _Hits(C.Structure):  # mm_b200_hits_t
    _fields_ = [("n_hits", C.c_int64), ("n_cigar", C.c_int64), ("n_str", C.c_int64), ("rows", C.POINTER(C.c_int64)),
                ("cigar", C.POINTER(C.c_uint32)), ("str", C.c_void_p)]


_lib = None
_lib_mu = threading.Lock()


def _L():
    global _lib
    with _lib_mu:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise ImportError(f"{LIB_PATH} missing: run `make` (the CUDA library is the mapper; there is no CPU fallback)")
            L = C.CDLL(LIB_PATH)
            P, I, U = C.c_void_p, C.c_int, C.c_char_p
            sig = {
                "mm_set_opt": (I, [U, C.POINTER(IdxOpt), C.POINTER(MapOpt)]),
                "mm_mapopt_update": (None, [C.POINTER(MapOpt), P]),
                "mm_b200_opt_error": (U, [C.POINTER(MapOpt)]),
                "mmg_device_count": (I, []),
                "mm_idx_reader_open": (P, [U, C.POINTER(IdxOpt), U]),
                "mm_idx_reader_read": (P, [P, I]),
                "mm_idx_reader_close": (None, [P]),
                "mm_idx_str": (P, [I, I, I, I, I, C.POINTER(U), C.POINTER(U)]),
                "mm_idx_destroy": (None, [P]),
                "mm_idx_name2id": (I, [P, U]),
                "mm_idx_getseq": (I, [P, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint8)]),
                "mm_b200_idx_seq": (I, [P, I, C.POINTER(U), C.POINTER(C.c_uint32)]),
                "mm_b200_map_hits": (C.POINTER(_Hits), [P, C.POINTER(MapOpt), I, C.POINTER(I), C.POINTER(U), U, I]),
                "mm_b200_batch_hits_flat": (C.POINTER(_Hits), [P, P, I]),
                "mm_b200_hits_free": (None, [C.POINTER(_Hits)]),
                "mm_b200_make_batch": (P, [I, C.POINTER(I), C.POINTER(I), C.POINTER(U), C.POINTER(U)]),
                "mm_b200_map_batches": (I, [P, C.POINTER(MapOpt), I, C.POINTER(P), I, I]),
                "mm_b200_free_batch": (None, [P]),
                "mm_fastx_open": (P, [U, I]),
                "mm_fastx_read": (I, [P, C.POINTER(U), C.POINTER(U), C.POINTER(U), C.POINTER(U)]),
                "mm_fastx_close": (None, [P]),
            }
            for name, (res, args) in sig.items():
                f = getattr(L, name)
                f.restype, f.argtypes = res, args
            _lib = L
        return _lib


def verbose(v=None):
    """the library's verbosity (mm_verbose); sets it first when v is given"""
    x = C.c_int.in_dll(_L(), "mm_verbose")
    if v is not None:
        x.value = v
    return x.value


_COMP = str.maketrans("ACGTUMRWSYKVHDBNacgtumrwsykvhdbn", "TGCAAKYWSRMBDHVNtgcaakywsrmbdhvn")  # seq_comp_table (misc.c)


def revcomp(seq):
    """the reverse complement of seq; IUPAC codes are complemented and case is kept, other characters stay as they are"""
    return None if seq is None else seq.translate(_COMP)[::-1]


def _str(p):
    return None if p is None else p.decode(errors="surrogateescape")


def fastx_read(fn, read_comment=False):
    """the records of a FASTA/FASTQ file, gzip'd or not: (name, seq, qual) or, with read_comment, (name, seq, qual, comment); qual
    and comment are None where the record has none.  A file that cannot be opened yields nothing, as in the reference."""
    L = _L()
    fp = L.mm_fastx_open(os.fsencode(fn), 1 if read_comment else 0)
    if not fp:
        return
    try:
        name, seq, qual, comment = C.c_char_p(), C.c_char_p(), C.c_char_p(), C.c_char_p()
        while L.mm_fastx_read(fp, C.byref(name), C.byref(seq), C.byref(qual), C.byref(comment)) >= 0:
            rec = (_str(name.value), _str(seq.value), _str(qual.value) or None)
            yield rec + (_str(comment.value),) if read_comment else rec
    finally:
        L.mm_fastx_close(fp)


class ThreadBuffer:
    """accepted for compatibility: every call keeps its own per-call state"""


class Alignment:
    """one hit; coordinates are 0-based, ends exclusive"""
    __slots__ = ("ctg", "ctg_len", "r_st", "r_en", "strand", "q_st", "q_en", "mapq", "cigar", "is_primary", "mlen", "blen", "NM",
                 "trans_strand", "read_num", "cs", "MD")

    def __init__(self, ctg, ctg_len, r_st, r_en, strand, q_st, q_en, mapq, cigar, is_primary, mlen, blen, NM, trans_strand,
                 read_num, cs, MD):
        self.ctg, self.ctg_len, self.r_st, self.r_en, self.strand = ctg, ctg_len, r_st, r_en, strand
        self.q_st, self.q_en, self.mapq, self.cigar, self.is_primary = q_st, q_en, mapq, cigar, is_primary
        self.mlen, self.blen, self.NM, self.trans_strand, self.read_num, self.cs, self.MD = mlen, blen, NM, trans_strand, read_num, cs, MD

    @property
    def cigar_str(self):
        return "".join(f"{n}{'MIDNSHP=XB'[op]}" for n, op in self.cigar)

    def __eq__(self, other):
        return isinstance(other, Alignment) and all(getattr(self, f) == getattr(other, f) for f in self.__slots__)

    def __repr__(self):
        return f"Alignment({', '.join(f'{f}={getattr(self, f)!r}' for f in self.__slots__)})"

    def __str__(self):
        ts = "ts:A:+" if self.trans_strand == 1 else "ts:A:-" if self.trans_strand == 2 else "ts:A:."
        a = [str(self.q_st), str(self.q_en), "+" if self.strand > 0 else "-", self.ctg, str(self.ctg_len), str(self.r_st),
             str(self.r_en), str(self.mlen), str(self.blen), str(self.mapq), "tp:A:P" if self.is_primary else "tp:A:S", ts,
             "cg:Z:" + self.cigar_str]
        if self.cs:
            a.append("cs:Z:" + self.cs)
        if self.MD:
            a.append("MD:Z:" + self.MD)
        return "\t".join(a)


class _SharedLock:
    """any number of shared holders, or one exclusive holder"""

    def __init__(self):
        self._cv = threading.Condition()
        self._shared = 0
        self._excl = False

    def acquire(self, exclusive):
        with self._cv:
            while self._excl or (exclusive and self._shared):
                self._cv.wait()
            if exclusive:
                self._excl = True
            else:
                self._shared += 1

    def release(self, exclusive):
        with self._cv:
            if exclusive:
                self._excl = False
            else:
                self._shared -= 1
            self._cv.notify_all()


def _enc(s):
    return s if isinstance(s, bytes) else s.encode()


def set_options(preset=None, k=None, w=None, min_cnt=None, min_chain_score=None, min_dp_score=None, bw=None, best_n=None,
                max_frag_len=None, extra_flags=None, scoring=None):
    """(mm_idxopt_t, mm_mapopt_t) as Aligner sets them up, in the reference mappy's order: mm_set_opt(NULL), the preset, MM_F_CIGAR,
    the whole reference as one index part, then the overrides.  Raises ValueError for an unknown preset and for options this
    build refuses (the library's message)."""
    L = _L()
    io, mo = IdxOpt(), MapOpt()
    L.mm_set_opt(None, C.byref(io), C.byref(mo))
    if preset is not None and L.mm_set_opt(_enc(preset), C.byref(io), C.byref(mo)) < 0:
        raise ValueError(f"unknown preset '{preset}'")
    mo.flag |= MM_F_CIGAR
    io.batch_size = 0x7fffffffffffffff  # the whole reference as one index part
    if k is not None:
        io.k = k
    if w is not None:
        io.w = w
    if min_cnt is not None:
        mo.min_cnt = min_cnt
    if min_chain_score is not None:
        mo.min_chain_score = min_chain_score
    if min_dp_score is not None:
        mo.min_dp_max = min_dp_score
    if bw is not None:
        mo.bw = bw
    if best_n is not None:
        mo.best_n = best_n
    if max_frag_len is not None:
        mo.max_frag_len = max_frag_len
    if extra_flags is not None:
        mo.flag |= extra_flags
    if scoring is not None and len(scoring) >= 4:
        mo.a, mo.b, mo.q, mo.e = scoring[0], scoring[1], scoring[2], scoring[3]
        mo.q2, mo.e2 = mo.q, mo.e
        if len(scoring) >= 6:
            mo.q2, mo.e2 = scoring[4], scoring[5]
            if len(scoring) >= 7:
                mo.sc_ambi = scoring[6]
    err = L.mm_b200_opt_error(C.byref(mo))
    if err:
        raise ValueError(err.decode())
    return io, mo


class Aligner:
    """An index on the GPU and the options to map against it (set_options: the preset, then the keyword overrides; scoring is
    [a,b,q,e], [a,b,q,e,q2,e2] or the same plus sc_ambi), then mm_mapopt_update.  The index is read from fn_idx_in (FASTA/FASTQ, gzip'd or not, or a .mmi; fn_idx_out writes
    the .mmi) or built from the one sequence seq.  bool(aligner) is False when no index could be read.

    Raises ValueError for options this build refuses, with the library's message, and RuntimeError without a CUDA device.

    map() may be called from any number of threads at once.  map_batch() maps on the index alone: mm_map_frag and the batch
    path must not map on one index at the same time, so map_batch waits for running map() calls and holds new ones back while
    it runs.  close() waits for both."""

    def __init__(self, fn_idx_in=None, preset=None, k=None, w=None, min_cnt=None, min_chain_score=None, min_dp_score=None, bw=None,
                 best_n=None, n_threads=3, fn_idx_out=None, max_frag_len=None, extra_flags=None, seq=None, scoring=None):
        self._idx = None
        self._lock = _SharedLock()
        L = _L()
        io, mo = set_options(preset, k, w, min_cnt, min_chain_score, min_dp_score, bw, best_n, max_frag_len, extra_flags, scoring)
        self._idx_opt, self._map_opt = io, mo
        if L.mmg_device_count() < 1:
            raise RuntimeError("no CUDA device: this mapper has no CPU path")
        if seq is None:
            if fn_idx_in is None:
                return
            rd = L.mm_idx_reader_open(os.fsencode(fn_idx_in), C.byref(io), os.fsencode(fn_idx_out) if fn_idx_out else None)
            if not rd:
                return
            self._idx = L.mm_idx_reader_read(rd, n_threads)
            L.mm_idx_reader_close(rd)
        else:
            self._idx = L.mm_idx_str(io.w, io.k, io.flag & MM_I_HPC, io.bucket_bits, 1, (C.c_char_p * 1)(_enc(seq)), None)
        if not self._idx:
            self._idx = None
            return
        L.mm_mapopt_update(C.byref(mo), self._idx)
        n = C.cast(self._idx, C.POINTER(_IdxHead)).contents.n_seq
        self._names, self._lens = [], []
        for i in range(n):
            nm, ln = C.c_char_p(), C.c_uint32()
            L.mm_b200_idx_seq(self._idx, i, C.byref(nm), C.byref(ln))
            self._names.append(_str(nm.value))
            self._lens.append(ln.value)

    def __bool__(self):
        return self._idx is not None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        self.close()

    def close(self):
        """frees the index once running calls have returned"""
        lock = getattr(self, "_lock", None)
        if lock is None:
            return
        lock.acquire(True)
        try:
            if self._idx is not None:
                _L().mm_idx_destroy(self._idx)
                self._idx = None
        finally:
            lock.release(True)

    def _head(self):
        return C.cast(self._idx, C.POINTER(_IdxHead)).contents

    @property
    def k(self):
        return self._head().k if self._idx is not None else None

    @property
    def w(self):
        return self._head().w if self._idx is not None else None

    @property
    def n_seq(self):
        return len(self._names) if self._idx is not None else 0

    @property
    def seq_names(self):
        return list(self._names) if self._idx is not None else None

    def seq(self, name, start=0, end=0x7fffffff):
        """the target's bases [start, end) in upper case ACGTN, from the host copy of the index; None for an unknown name or an
        empty range"""
        if self._idx is None:
            return None
        L = _L()
        rid = L.mm_idx_name2id(self._idx, _enc(name))
        if rid < 0:
            return None
        end = min(end, self._lens[rid])
        if start < 0 or start >= end:
            return None
        buf = (C.c_uint8 * (end - start))()
        if L.mm_idx_getseq(self._idx, rid, start, end, buf) < 0:
            return None
        return bytes(buf).translate(bytes.maketrans(bytes(range(5)), b"ACGTN")).decode()

    def _opt(self, max_frag_len, extra_flags):
        if max_frag_len is None and extra_flags is None:
            return self._map_opt
        o = MapOpt()
        C.memmove(C.byref(o), C.byref(self._map_opt), C.sizeof(o))
        if max_frag_len is not None:
            o.max_frag_len = max_frag_len
        if extra_flags is not None:
            o.flag |= extra_flags
        err = _L().mm_b200_opt_error(C.byref(o))
        if err:
            raise ValueError(err.decode())
        return o

    def _alignments(self, hp, reads):
        """Alignment lists of the fragments of a hits block; reads[f] holds the reads of fragment f"""
        L = _L()
        h = hp.contents
        n, cols = h.n_hits, MM_B200_HITS_COLS
        rows = h.rows[:n * cols] if n else []
        cig = h.cigar[:h.n_cigar] if h.n_cigar else []
        strs = C.string_at(h.str, h.n_str) if h.n_str else b""
        out = [[] for _ in reads]
        for i in range(0, n * cols, cols):
            r = rows[i:i + cols]
            rid = r[_RID]
            c0 = r[_CIGAR_OFF]
            cigar = [[x >> 4, x & 0xf] for x in cig[c0:c0 + r[_N_CIGAR]]]
            cs = strs[r[_CS_OFF]:r[_CS_OFF] + r[_CS_LEN]].decode() if r[_CS_OFF] >= 0 else ""
            md = strs[r[_MD_OFF]:r[_MD_OFF] + r[_MD_LEN]].decode() if r[_MD_OFF] >= 0 else ""
            ctg = self._names[rid]
            out[r[_FRAG]].append(Alignment(ctg if ctg is not None else str(rid), self._lens[rid], r[_RS], r[_RE], -1 if r[_REV] else 1,
                                           r[_QS], r[_QE], r[_MAPQ], cigar, bool(r[_PRI]), r[_MLEN], r[_BLEN],
                                           r[_BLEN] - r[_MLEN] + r[_N_AMBI], r[_TS], r[_SEG] + 1, cs, md))
        L.mm_b200_hits_free(hp)
        return out

    def map(self, seq, seq2=None, buf=None, cs=False, MD=False, max_frag_len=None, extra_flags=None, name=None):
        """The hits of seq, or of the pair (seq, seq2), as Alignments.  seq2 is given as sequenced: it is mapped as its reverse
        complement and its hits are reported in its own orientation.  cs gives the short cs string (--cs), MD the MD string.
        buf (a ThreadBuffer) is accepted and not needed.  name seeds the choice among equally good chains as a read name does."""
        if self._idx is None:
            return
        opt = self._opt(max_frag_len, extra_flags)
        segs = [_enc(seq)] if seq2 is None else [_enc(seq), _enc(seq2)]
        flags = (MM_B200_HITS_CS if cs else 0) | (MM_B200_HITS_MD if MD else 0)
        self._lock.acquire(False)
        try:
            if self._idx is None:
                return
            hp = _L().mm_b200_map_hits(self._idx, C.byref(opt), len(segs), (C.c_int * len(segs))(*map(len, segs)),
                                       (C.c_char_p * len(segs))(*segs), _enc(name) if name is not None else None, flags)
        finally:
            self._lock.release(False)
        yield from self._alignments(hp, [segs])[0]

    def map_batch(self, reads, cs=False, MD=False, names=None):
        """The hits of every entry of reads (a sequence, or a pair (seq, seq2) given as map() takes it), as one list of
        Alignments per entry, in input order.  The reads are cut into mini-batches of mini_batch_size bases and mapped with
        mm_b200_map_batches, two mini-batches in flight; the hits equal those of map() on each entry.  names: one read name per
        entry, or None.

        The batch path and mm_map_frag must not map on the same index at the same time: this call waits for running map()
        calls, and map() calls made meanwhile wait for it."""
        if self._idx is None:
            return [[] for _ in reads]
        L = _L()
        frags = [[_enc(r)] if isinstance(r, (str, bytes)) else [_enc(x) for x in r] for r in reads]
        if any(not 1 <= len(f) <= 2 for f in frags):
            raise ValueError("an entry of reads is a sequence or a pair of sequences")
        if names is not None and len(names) != len(frags):
            raise ValueError("names must give one name per entry of reads")
        opt = MapOpt()
        C.memmove(C.byref(opt), C.byref(self._map_opt), C.sizeof(opt))
        if opt.pe_ori >= 0:
            opt.pe_ori = 1  # read 2 mapped as its reverse complement, as map() maps it
        opt.flag &= ~MM_F_INDEPEND_SEG  # the reads of a pair mapped jointly, as map() maps them
        flags = (MM_B200_HITS_CS if cs else 0) | (MM_B200_HITS_MD if MD else 0)
        cuts, acc = [0], 0
        for i, f in enumerate(frags):  # mini-batches as the file reader cuts them: close one once it holds enough bases
            acc += sum(map(len, f))
            if acc >= opt.mini_batch_size:
                cuts.append(i + 1)
                acc = 0
        if cuts[-1] != len(frags):
            cuts.append(len(frags))
        out = []
        self._lock.acquire(True)
        batches = []
        try:
            if self._idx is None:
                return [[] for _ in reads]
            for b0, b1 in zip(cuts[:-1], cuts[1:]):
                part = frags[b0:b1]
                segs = [s for f in part for s in f]
                nm = None if names is None else (C.c_char_p * len(part))(*[_enc(x) if x is not None else None for x in names[b0:b1]])
                b = L.mm_b200_make_batch(len(part), (C.c_int * len(part))(*map(len, part)), (C.c_int * len(segs))(*map(len, segs)),
                                         (C.c_char_p * len(segs))(*segs), nm)
                if not b:
                    raise MemoryError("cannot stage the reads")
                batches.append(b)
            if batches and L.mm_b200_map_batches(self._idx, C.byref(opt), os.cpu_count() or 1, (C.c_void_p * len(batches))(*batches),
                                                 len(batches), 0) != 0:
                raise RuntimeError("mapping failed")
            for (b0, b1), b in zip(zip(cuts[:-1], cuts[1:]), batches):
                out += self._alignments(L.mm_b200_batch_hits_flat(self._idx, b, flags), frags[b0:b1])
        finally:
            for b in batches:
                L.mm_b200_free_batch(b)
            self._lock.release(True)
        return out
