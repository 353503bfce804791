"""ctypes binding of include/mmg.h (libmm2b200.so).

Python is only a harness here (tests, bench.py); the product is the C library.  The library is
loaded from this package directory and the import FAILS LOUDLY when it is missing: there is no
CPU fallback anywhere behind this module.
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmm2b200.so")

mm128 = np.dtype([("x", "<u8"), ("y", "<u8")])

MM_F_CIGAR = 0x004
MM_F_OUT_SAM = 0x008
MM_F_SPLICE = 0x080
MM_F_SR = 0x1000
MM_F_FRAG_MODE = 0x2000
MM_F_NO_PRINT_2ND = 0x4000
MM_F_2_IO_THREADS = 0x8000
MM_F_FOR_ONLY = 0x100000
MM_F_REV_ONLY = 0x200000
MM_F_HEAP_SORT = 0x400000
MM_F_NO_DIAG = 0x001
MM_F_NO_DUAL = 0x002
NAME_NONE = 0xffffffff  # MMG_NAME_NONE: the unit key of a fragment without a name


class MmgError(RuntimeError):
    pass


class Extz(C.Structure):
    _fields_ = [("max", C.c_uint32), ("zdropped", C.c_int32), ("max_q", C.c_int32), ("max_t", C.c_int32), ("mqe", C.c_int32),
                ("mqe_t", C.c_int32), ("mte", C.c_int32), ("mte_q", C.c_int32), ("score", C.c_int32), ("n_cigar", C.c_int32),
                ("reach_end", C.c_int32)]


class MapOpt(C.Structure):  # mmg_mapopt_t
    _fields_ = [("flag", C.c_int64), ("mid_occ", C.c_int32), ("max_occ", C.c_int32), ("bw", C.c_int32), ("max_gap", C.c_int32),
                ("max_gap_ref", C.c_int32), ("max_frag_len", C.c_int32), ("max_chain_skip", C.c_int32), ("max_chain_iter", C.c_int32),
                ("min_cnt", C.c_int32), ("min_chain_score", C.c_int32), ("pe_ori", C.c_int32), ("a", C.c_int32), ("b", C.c_int32),
                ("q", C.c_int32), ("e", C.c_int32), ("q2", C.c_int32), ("e2", C.c_int32), ("sc_ambi", C.c_int32)]


class Batch(C.Structure):  # mmg_batch_t
    _fields_ = [("n_frag", C.c_int32), ("n_seq", C.c_int32), ("n_seg", C.c_void_p), ("seg_off", C.c_void_p), ("seq_len", C.c_void_p),
                ("seq_off", C.c_void_p), ("bases", C.c_void_p), ("n_bases", C.c_uint64), ("flip", C.c_void_p), ("ukey", C.c_void_p)]


class Chains(C.Structure):  # mmg_chains_t
    _fields_ = [("n_frag", C.c_int32), ("n_u", C.POINTER(C.c_int32)), ("n_a", C.POINTER(C.c_int32)), ("rep_len", C.POINTER(C.c_int32)),
                ("n_mini", C.POINTER(C.c_int32)), ("rechained", C.POINTER(C.c_int32)), ("u_off", C.POINTER(C.c_uint64)),
                ("a_off", C.POINTER(C.c_uint64)), ("mini_off", C.POINTER(C.c_uint64)), ("u", C.POINTER(C.c_uint64)),
                ("a", C.c_void_p), ("mini_pos", C.POINTER(C.c_uint64)), ("t_h2d_ms", C.c_double), ("t_kernels_ms", C.c_double),
                ("t_d2h_ms", C.c_double), ("n_minimizers", C.c_uint64), ("n_anchors", C.c_uint64), ("n_chain_iter", C.c_uint64)]


class KswJob(C.Structure):  # mmg_ksw_job_t
    _fields_ = [("seq_id", C.c_int32), ("q_rev", C.c_int32), ("q_start", C.c_int32), ("q_len", C.c_int32), ("rid", C.c_int32),
                ("t_start", C.c_int32), ("t_len", C.c_int32), ("reversed", C.c_int32), ("w", C.c_int32), ("zdrop", C.c_int32),
                ("end_bonus", C.c_int32), ("flag", C.c_int32)]


class KswRes(C.Structure):  # mmg_ksw_res_t
    _fields_ = [("ez", Extz), ("cigar_off", C.c_uint64)]


ksw_job_dtype = np.dtype([(n, "<i4") for n in ["seq_id", "q_rev", "q_start", "q_len", "rid", "t_start", "t_len", "reversed", "w",
                                                "zdrop", "end_bonus", "flag"]])

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MmgError(f"{LIB_PATH} is missing: run `make lib` (nvcc, sm_100a). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        L.mmg_last_error.restype = C.c_char_p
        L.mmg_init.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.mmg_destroy.argtypes = [C.c_void_p]
        L.mmg_launch_count.restype = C.c_long
        L.mmg_launch_count.argtypes = [C.c_void_p, C.c_int]
        L.mmg_stream.restype = C.c_void_p
        L.mmg_stream.argtypes = [C.c_void_p]
        L.mmg_idx_build.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_char_p), C.c_void_p, C.POINTER(C.c_void_p)]
        L.mmg_idx_free.argtypes = [C.c_void_p]
        for f in ("mmg_idx_n_minimizers", "mmg_idx_n_keys"):
            getattr(L, f).restype = C.c_int64
            getattr(L, f).argtypes = [C.c_void_p]
        L.mmg_idx_total_len.restype = C.c_uint64
        L.mmg_idx_total_len.argtypes = [C.c_void_p]
        L.mmg_idx_bytes.restype = C.c_size_t
        L.mmg_idx_bytes.argtypes = [C.c_void_p]
        L.mmg_idx_copy_S.argtypes = [C.c_void_p, C.c_void_p]
        L.mmg_idx_cal_max_occ.argtypes = [C.c_void_p, C.c_float, C.POINTER(C.c_int32)]
        L.mmg_idx_get.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.mmg_idx_clone_to.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
        L.mmg_sketch.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.mmg_collect_seeds.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                        C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p]
        L.mmg_chain_dp.argtypes = [C.c_void_p] + [C.c_int] * 9 + [C.c_int64, C.c_void_p, C.POINTER(C.c_int), C.c_void_p]
        L.mmg_ksw_extd2.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int8, C.c_void_p, C.c_int8, C.c_int8,
                                    C.c_int8, C.c_int8, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(Extz), C.c_void_p]
        L.mmg_seed_chain_batch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(MapOpt), C.POINTER(Batch), C.POINTER(Chains)]
        L.mmg_batch_upload.argtypes = [C.c_void_p, C.POINTER(MapOpt), C.POINTER(Batch)]
        L.mmg_seed_chain_resident.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(MapOpt), C.POINTER(Chains), C.c_int]
        L.mmg_collect_seeds_named.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_uint32,
                                              C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p]
        L.mmg_idx_set_name_keys.argtypes = [C.c_void_p, C.c_void_p]
        L.mm_b200_name_order.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.c_void_p]
        L.mm_b200_name_ukey.restype = C.c_uint32
        L.mm_b200_name_ukey.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.c_char_p]
        L.mmg_path_counts.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.mmg_ksw_batch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(MapOpt), C.c_int, C.c_void_p, C.c_void_p,
                                    C.POINTER(C.POINTER(C.c_uint32)), C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise MmgError(f"mmg error {rc}: {lib().mmg_last_error().decode()}")


def sr_opt(cigar=True):
    """`-x sr` (options.c:105-122) as seen by the device stages."""
    o = MapOpt()
    o.flag = MM_F_SR | MM_F_FRAG_MODE | MM_F_NO_PRINT_2ND | MM_F_2_IO_THREADS | MM_F_HEAP_SORT | (MM_F_CIGAR if cigar else 0)
    o.mid_occ, o.max_occ = 1000, 5000
    o.bw, o.max_gap, o.max_gap_ref, o.max_frag_len = 100, 100, -1, 800
    o.max_chain_skip, o.max_chain_iter, o.min_cnt, o.min_chain_score = 25, 5000, 2, 25
    o.pe_ori = 1
    o.a, o.b, o.q, o.e, o.q2, o.e2, o.sc_ambi = 2, 8, 12, 2, 24, 1, 1
    return o


def ont_opt(mid_occ, cigar=True):
    """`-x map-ont` (options.c:13-49,85-86); mid_occ comes from mmg_idx_cal_max_occ(2e-4)."""
    o = MapOpt()
    o.flag = MM_F_CIGAR if cigar else 0
    o.mid_occ, o.max_occ = mid_occ, 0
    o.bw, o.max_gap, o.max_gap_ref, o.max_frag_len = 500, 5000, -1, 0
    o.max_chain_skip, o.max_chain_iter, o.min_cnt, o.min_chain_score = 25, 5000, 3, 40
    o.pe_ori = 0
    o.a, o.b, o.q, o.e, o.q2, o.e2, o.sc_ambi = 2, 4, 4, 2, 24, 1, 1
    return o


class Context:
    def __init__(self, device=0):
        self.h = C.c_void_p()
        _check(lib().mmg_init(device, C.byref(self.h)))

    def close(self):
        if self.h:
            lib().mmg_destroy(self.h)
            self.h = C.c_void_p()

    def launches(self, reset=False):
        return lib().mmg_launch_count(self.h, 1 if reset else 0)

    def stream(self):
        return lib().mmg_stream(self.h)

    # -- per-kernel entry points
    def sketch(self, seq: bytes, w, k, rid=0, hpc=0):
        out = np.zeros(len(seq) + 8, dtype=mm128)
        n = C.c_int(0)
        _check(lib().mmg_sketch(self.h, seq, len(seq), w, k, rid, hpc, out.ctypes.data, len(out), C.byref(n)))
        return out[:n.value].copy()

    def collect_seeds(self, idx, heap_sort, flag, max_occ, mv, qlen, cap, name=False):
        """name: the fragment's name (bytes, or None for no name) against an Index whose set_names() was called; False: no
        self/dual filtering (mmg_collect_seeds)"""
        mv = np.ascontiguousarray(mv)
        a = np.zeros(cap + 1, dtype=mm128)
        mp = np.zeros(len(mv) + 1, dtype=np.uint64)
        n_a, rep, nm = C.c_int64(0), C.c_int(0), C.c_int(0)
        if name is False:
            _check(lib().mmg_collect_seeds(self.h, idx.h, int(heap_sort), flag, max_occ, len(mv), mv.ctypes.data, qlen, a.ctypes.data, cap,
                                           C.byref(n_a), C.byref(rep), C.byref(nm), mp.ctypes.data))
        else:
            _check(lib().mmg_collect_seeds_named(self.h, idx.h, int(heap_sort), flag, max_occ, len(mv), mv.ctypes.data, qlen, idx.unit_key(name),
                                                 a.ctypes.data, cap, C.byref(n_a), C.byref(rep), C.byref(nm), mp.ctypes.data))
        return a[:n_a.value].copy(), rep.value, mp[:nm.value].copy()

    def path_counts(self, reset=False):
        out = np.zeros(8, dtype=np.uint64)
        lib().mmg_path_counts(self.h, out.ctypes.data, 1 if reset else 0)
        return out

    def chain_dp(self, params, a):
        a = np.ascontiguousarray(a.copy())
        u = np.zeros(len(a) + 1, dtype=np.uint64)
        n_u = C.c_int(0)
        _check(lib().mmg_chain_dp(self.h, *params, len(a), a.ctypes.data, C.byref(n_u), u.ctypes.data))
        u = u[:n_u.value].copy()
        return u, a[:int((u & np.uint64(0xffffffff)).sum())].copy()

    def ksw_extd2(self, q, t, mat, gq, ge, gq2, ge2, w, zdrop, end_bonus, flag):
        q = np.ascontiguousarray(q, dtype=np.uint8)
        t = np.ascontiguousarray(t, dtype=np.uint8)
        ez = Extz()
        cig = np.zeros(len(q) + len(t) + 4, dtype=np.uint32)
        _check(lib().mmg_ksw_extd2(self.h, len(q), q.ctypes.data, len(t), t.ctypes.data, 5, mat.ctypes.data, gq, ge, gq2, ge2, w, zdrop,
                                   end_bonus, flag, C.byref(ez), cig.ctypes.data))
        return dict(max=ez.max, zdropped=ez.zdropped, max_q=ez.max_q, max_t=ez.max_t, mqe=ez.mqe, mqe_t=ez.mqe_t, mte=ez.mte,
                    mte_q=ez.mte_q, score=ez.score, reach_end=ez.reach_end, cigar=cig[:ez.n_cigar].tolist())

    # -- batched stages
    @staticmethod
    def make_batch(frags):
        """frags: list of lists of bytes (segments, original orientation). Returns (Batch, keepalive)."""
        seqs = [s for f in frags for s in f]
        n_seg = np.array([len(f) for f in frags], dtype=np.int32)
        seg_off = np.concatenate([[0], np.cumsum(n_seg)[:-1]]).astype(np.int32) if len(frags) else np.zeros(0, np.int32)
        seq_len = np.array([len(s) for s in seqs], dtype=np.int32)
        seq_off = np.concatenate([[0], np.cumsum(seq_len.astype(np.uint64))[:-1]]).astype(np.uint64) if len(seqs) else np.zeros(0, np.uint64)
        bases = np.frombuffer(b"".join(seqs), dtype=np.uint8).copy() if seqs else np.zeros(1, np.uint8)
        b = Batch(len(frags), len(seqs), n_seg.ctypes.data, seg_off.ctypes.data, seq_len.ctypes.data, seq_off.ctypes.data,
                  bases.ctypes.data, int(seq_len.sum()))
        return b, (n_seg, seg_off, seq_len, seq_off, bases)

    def seed_chain_batch(self, idx, opt, batch):
        out = Chains()
        _check(lib().mmg_seed_chain_batch(self.h, idx.h, C.byref(opt), C.byref(batch), C.byref(out)))
        return out

    def batch_upload(self, opt, batch, flips=None, names=None, idx=None):
        """flips: None (mates flipped per opt.pe_ori within each fragment) or one 0/1 per read: 1 = reverse-complemented before
        mapping, whatever fragment the read is in (how --no-pairing maps the mates of a pair one by one).
        names: one name (bytes, or None) per fragment for the self/dual filters (-D, --dual=no), ordered against the target names
        given to idx.set_names()."""
        b = Batch.from_buffer_copy(batch)  # the caller's batch keeps no pointer into the arrays made here
        if flips is not None:
            flips = np.ascontiguousarray(flips, dtype=np.uint8)
            if len(flips) != batch.n_seq:
                raise ValueError(f"{len(flips)} flips for {batch.n_seq} reads")
            b.flip = flips.ctypes.data
        if names is not None:
            if idx is None or len(names) != batch.n_frag:
                raise ValueError("names needs one name per fragment and the Index they are ordered against")
            ukey = np.array([idx.unit_key(n) for n in names], dtype=np.uint32)
            b.ukey = ukey.ctypes.data
        _check(lib().mmg_batch_upload(self.h, C.byref(opt), C.byref(b)))

    def seed_chain_resident(self, idx, opt, download=True):
        out = Chains()
        _check(lib().mmg_seed_chain_resident(self.h, idx.h, C.byref(opt), C.byref(out), 1 if download else 0))
        return out

    def ksw_batch(self, idx, opt, jobs):
        """jobs: numpy array of ksw_job_dtype. Returns (list of dict results, kernel_ms, cells)."""
        jobs = np.ascontiguousarray(jobs)
        n = len(jobs)
        res = (KswRes * max(n, 1))()
        cig = C.POINTER(C.c_uint32)()
        ms, cells = C.c_double(0), C.c_uint64(0)
        _check(lib().mmg_ksw_batch(self.h, idx.h, C.byref(opt), n, jobs.ctypes.data, res, C.byref(cig), C.byref(ms), C.byref(cells)))
        out = []
        for i in range(n):
            ez = res[i].ez
            o = res[i].cigar_off
            out.append(dict(max=ez.max, zdropped=ez.zdropped, max_q=ez.max_q, max_t=ez.max_t, mqe=ez.mqe, mqe_t=ez.mqe_t, mte=ez.mte,
                            mte_q=ez.mte_q, score=ez.score, reach_end=ez.reach_end, cigar=[cig[o + j] for j in range(ez.n_cigar)]))
        return out, ms.value, cells.value


class Index:
    def __init__(self, ctx, seqs, w, k, hpc=0):
        self.ctx = ctx
        self.h = C.c_void_p()
        arr = (C.c_char_p * len(seqs))(*seqs)
        lens = np.array([len(s) for s in seqs], dtype=np.uint32)
        _check(lib().mmg_idx_build(ctx.h, w, k, hpc, len(seqs), arr, lens.ctypes.data, C.byref(self.h)))
        self.w, self.k = w, k

    def close(self):
        if self.h:
            lib().mmg_idx_free(self.h)
            self.h = C.c_void_p()

    def set_names(self, names):
        """the targets' names (bytes, one per sequence): computes and uploads their name keys for the self/dual filters"""
        n = len(names)
        self._names = (C.c_char_p * max(n, 1))(*names)  # the sorted table points into these
        self._sorted = (C.c_char_p * max(n, 1))()
        tkey = np.zeros(max(n, 1), dtype=np.uint32)
        lib().mm_b200_name_order(n, self._names, self._sorted, tkey.ctypes.data)
        self._n_names = n
        _check(lib().mmg_idx_set_name_keys(self.h, tkey.ctypes.data))

    def unit_key(self, name):
        """the name key of a fragment named `name` (None: no name) against the names of set_names()"""
        return lib().mm_b200_name_ukey(self._n_names, self._sorted, name)

    def n_minimizers(self):
        return lib().mmg_idx_n_minimizers(self.h)

    def n_keys(self):
        return lib().mmg_idx_n_keys(self.h)

    def bytes(self):
        return lib().mmg_idx_bytes(self.h)

    def packed_S(self):
        n = lib().mmg_idx_total_len(self.h)
        S = np.zeros((n + 7) // 8, dtype=np.uint32)
        _check(lib().mmg_idx_copy_S(self.h, S.ctypes.data))
        return S

    def cal_max_occ(self, f):
        t = C.c_int32(0)
        _check(lib().mmg_idx_cal_max_occ(self.h, f, C.byref(t)))
        return t.value

    def get(self, miniers, max_pos):
        q = np.ascontiguousarray(miniers, dtype=np.uint64)
        n = np.zeros(len(q), dtype=np.int32)
        pos = np.zeros((len(q), max(max_pos, 1)), dtype=np.uint64)
        _check(lib().mmg_idx_get(self.ctx.h, self.h, len(q), q.ctypes.data, n.ctypes.data, max_pos, pos.ctypes.data))
        return n, pos


def chains_to_py(ch: Chains):
    """Copy a mmg_chains_t into plain numpy arrays (the ctx-owned buffers are reused by the next call)."""
    nf = ch.n_frag
    g = lambda p, n, dt: np.ctypeslib.as_array(p, shape=(n,)).astype(dt).copy() if n else np.zeros(0, dt)
    n_u, n_a, rep, nmini, rech = (g(p, nf, np.int32) for p in (ch.n_u, ch.n_a, ch.rep_len, ch.n_mini, ch.rechained))
    u_off, a_off, m_off = (g(p, nf + 1, np.uint64) for p in (ch.u_off, ch.a_off, ch.mini_off))
    u = g(ch.u, int(u_off[-1]) if nf else 0, np.uint64)
    na_tot = int(a_off[-1]) if nf else 0
    a = np.zeros(na_tot, dtype=mm128)
    if na_tot:
        C.memmove(a.ctypes.data, ch.a, na_tot * 16)
    mini = g(ch.mini_pos, int(m_off[-1]) if nf else 0, np.uint64)
    return dict(n_u=n_u, n_a=n_a, rep_len=rep, n_mini=nmini, rechained=rech, u_off=u_off, a_off=a_off, mini_off=m_off, u=u, a=a, mini_pos=mini)
