#!/usr/bin/env python3
"""Reads/s of the per-fragment API (mm_map_frag, one call per read pair) from 1, 4, 16 and 64 caller threads, next to the batch
path (mm_b200_map_batches) on the same reads and, with --parent-lib, next to an earlier build's mm_map_frag from 1 and 16 threads.

The calls of concurrent threads are mapped together in shared mini-batches (airlift_b200/host/apiq.c); a build that maps one
fragment per call shows what that sharing gains.  The arms that make one device round trip per pair (one caller thread, and
every arm of --parent-lib) map the first --slow-pairs pairs only; every arm's hits are digested and must equal the batch path's
on the same pairs.  The ctypes arrays of every call are built before the timed region.  `caller_cpu_us_per_call` is the CPU time
of the Python caller threads per call: where it approaches wall time x threads / calls, Python, not the mapper, is the limit.
The card's name and power limit are read in the same run (nvidia-smi query only) and printed with the rates as one JSON line.
Needs a GPU and build/mmsynth."""
import argparse
import ctypes as C
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

MM_F_CIGAR, MM_F_OUT_SAM = 0x004, 0x008
libc = C.CDLL("libc.so.6")
libc.free.argtypes = [C.c_void_p]


class Extra(C.Structure):
    _fields_ = [("capacity", C.c_uint32), ("dp_score", C.c_int32), ("dp_max", C.c_int32), ("dp_max2", C.c_int32),
                ("n_ambi_ts", C.c_uint32), ("n_cigar", C.c_uint32)]


class Reg1(C.Structure):  # mm_reg1_t
    _fields_ = [(n, C.c_int32) for n in ("id", "cnt", "rid", "score", "qs", "qe", "rs", "re", "parent", "subsc", "as_", "mlen", "blen", "n_sub", "score0")] + \
               [("bits", C.c_uint32), ("hash", C.c_uint32), ("div", C.c_float), ("p", C.POINTER(Extra))]


class StepHead(C.Structure):
    _fields_ = [("n_seq", C.c_int), ("n_frag", C.c_int), ("seq", C.c_void_p), ("n_reg", C.POINTER(C.c_int)), ("seg_off", C.POINTER(C.c_int)),
                ("n_seg", C.POINTER(C.c_int)), ("rep_len", C.POINTER(C.c_int)), ("frag_gap", C.POINTER(C.c_int)), ("reg", C.POINTER(C.POINTER(Reg1)))]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    if q.returncode != 0:
        raise SystemExit("nvidia-smi failed: this measurement needs a GPU")
    name, power = [x.strip() for x in q.stdout.strip().split(",")]
    return {"name": name, "power_limit": power}


def hits(regs, n, flip_qlen=None):
    """the hits of one read as tuples; a mate mapped reverse-complemented is put back in its own orientation"""
    out = []
    for i in range(n):
        r = regs[i]
        qs, qe, rev = r.qs, r.qe, r.bits >> 10 & 1
        if flip_qlen is not None:
            qs, qe, rev = flip_qlen - r.qe, flip_qlen - r.qs, 1 - rev
        cig = ()
        if r.p:
            arr = C.cast(C.addressof(r.p.contents) + C.sizeof(Extra), C.POINTER(C.c_uint32))
            cig = tuple(arr[j] for j in range(r.p.contents.n_cigar))
        out.append((r.rid, r.rs, r.re, qs, qe, rev, r.bits & 0xff, r.score, r.p.contents.dp_max if r.p else -1, cig))
    return out


def digest(per_read):
    h = hashlib.sha256()
    for i, hs in enumerate(per_read):
        h.update(repr((i, hs)).encode())
    return h.hexdigest()[:16]


def load(path):
    L = bench.load_lib() if path is None else None
    if path is not None:  # an earlier build: same C ABI, loaded under its own handle
        saved = bench.LIB
        bench.LIB = path
        try:
            L = bench.load_lib()
        finally:
            bench.LIB = saved
    L.mm_map_frag.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_char_p), C.POINTER(C.c_int), C.POINTER(C.POINTER(Reg1)),
                              C.c_void_p, C.POINTER(bench.MapOptFull), C.c_char_p]
    L.mm_tbuf_init.restype = C.c_void_p
    L.mm_tbuf_destroy.argtypes = [C.c_void_p]
    L.mm_b200_set_lanes.argtypes = [C.c_int]
    return L


def index(L, ref):
    L.mm_b200_set_devices(1, (C.c_int * 1)(0))
    L.mm_b200_set_lanes(4)
    L.mm_b200_set_in_flight(2)
    ipt, opt = bench.IdxOpt(), bench.MapOptFull()
    L.mm_set_opt(None, C.byref(ipt), C.byref(opt))
    L.mm_set_opt(b"sr", C.byref(ipt), C.byref(opt))
    opt.flag |= MM_F_CIGAR | MM_F_OUT_SAM
    rd = L.mm_idx_reader_open(ref.encode(), C.byref(ipt), None)
    mi = L.mm_idx_reader_read(rd, 3)
    L.mm_idx_reader_close(rd)
    if not mi:
        raise SystemExit("index construction failed")
    L.mm_mapopt_update(C.byref(opt), mi)
    return mi, opt


def read_pairs(fn1, fn2):
    def rd(fn):
        ls = open(fn).read().split("\n")
        return [(ls[i][1:].split()[0], ls[i + 1]) for i in range(0, len(ls) - 3, 4)]
    return list(zip(rd(fn1), rd(fn2)))


_COMP = bytes.maketrans(b"ACGTN", b"TGCAN")


class Calls:
    """the ctypes arguments of one mm_map_frag call per pair, built once"""
    def __init__(self, pairs):
        self.n = len(pairs)
        self.names, self.seqs, self.qlens, self.n_regs, self.regs, self.l2 = [], [], [], [], [], []
        for (n1, s1), (_, s2) in pairs:
            s2rc = s2.encode().translate(_COMP)[::-1]
            self.names.append(n1.encode())
            self.seqs.append((C.c_char_p * 2)(s1.encode(), s2rc))
            self.qlens.append((C.c_int * 2)(len(s1), len(s2)))
            self.n_regs.append((C.c_int * 2)())
            self.regs.append((C.POINTER(Reg1) * 2)())
            self.l2.append(len(s2))

    def collect(self, n):
        """hits of the first n calls per read (mate 1, mate 2, ...), then their arrays are freed"""
        out = []
        for k in range(n):
            nr, rg = self.n_regs[k], self.regs[k]
            out.append(hits(rg[0], nr[0]))
            out.append(hits(rg[1], nr[1], flip_qlen=self.l2[k]))
            for j in range(2):
                for i in range(nr[j]):
                    libc.free(C.cast(rg[j][i].p, C.c_void_p))
                libc.free(C.cast(rg[j], C.c_void_p))
                nr[j] = 0
        return out


def run_api(L, mi, opt, calls, n, n_threads):
    """n calls spread over n_threads callers; returns wall seconds and caller CPU seconds"""
    optref = C.byref(opt)
    cpu = [0.0] * n_threads
    go = threading.Barrier(n_threads + 1)

    def work(t):
        tb = L.mm_tbuf_init()
        f = L.mm_map_frag
        go.wait()
        c0 = time.thread_time()
        for k in range(t, n, n_threads):
            f(mi, 2, calls.qlens[k], calls.seqs[k], calls.n_regs[k], calls.regs[k], tb, optref, calls.names[k])
        cpu[t] = time.thread_time() - c0
        L.mm_tbuf_destroy(tb)
    th = [threading.Thread(target=work, args=(t,)) for t in range(n_threads)]
    for t in th:
        t.start()
    go.wait()
    t0 = time.perf_counter()
    for t in th:
        t.join()
    return time.perf_counter() - t0, sum(cpu)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genome-bp", type=int, default=100_000_000)
    ap.add_argument("--contigs", type=int, default=4)
    ap.add_argument("--pairs", type=int, default=200_000)
    ap.add_argument("--slow-pairs", type=int, default=10_000, help="pairs of the arms that make one round trip per pair")
    ap.add_argument("--threads", default="1,4,16,64")
    ap.add_argument("--parent-lib", default=None, help="libmm2b200.so of an earlier build, for its mm_map_frag")
    args = ap.parse_args()
    card = gpu_info()
    bench.ensure_tools()
    cores = os.cpu_count() or 1
    d = tempfile.mkdtemp(prefix="api_tput_")
    try:
        ref, r1, r2 = (os.path.join(d, x) for x in ("ref.fa", "r1.fq", "r2.fq"))
        subprocess.check_call([bench.SYNTH, "ref", ref, str(args.genome_bp), str(args.contigs), "42"])
        subprocess.check_call([bench.SYNTH, "sr", ref, r1, r2, str(args.pairs), "44"])
        pairs = read_pairs(r1, r2)
        n_slow = min(args.slow_pairs, len(pairs))
        out = {"gpu": card, "cores": cores, "genome_bp": args.genome_bp, "pairs": len(pairs), "slow_pairs": n_slow,
               "preset": "-ax sr", "lanes": 4, "arms": {}}
        L = load(None)
        mi, opt = index(L, ref)

        # batch path: the same reads as mini-batches of opt.mini_batch_size bases, two in flight
        fns = (C.c_char_p * 2)(r1.encode(), r2.encode())
        reader = L.mm_b200_open_reads(2, fns)
        bs = []
        while True:
            b = L.mm_b200_read_batch(reader, C.byref(opt), opt.mini_batch_size)
            if not b:
                break
            bs.append(b)
        L.mm_b200_close_reads(reader)
        arr = (C.c_void_p * len(bs))(*bs)
        if L.mm_b200_map_batches(mi, C.byref(opt), cores, arr, len(bs), 0) != 0:  # warm: every buffer at its working size
            raise SystemExit("mapping failed")
        for b in bs:
            L.mm_b200_reset_batch(b)
        t0 = time.perf_counter()
        if L.mm_b200_map_batches(mi, C.byref(opt), cores, arr, len(bs), 0) != 0:
            raise SystemExit("mapping failed")
        t = time.perf_counter() - t0
        want = []
        for b in bs:
            h = C.cast(b, C.POINTER(StepHead)).contents
            want += [hits(h.reg[r], h.n_reg[r]) for r in range(h.n_seq)]
            L.mm_b200_free_batch(b)
        dig_all, dig_slow = digest(want), digest(want[:2 * n_slow])
        out["arms"]["map_batches"] = {"reads": len(want), "reads_per_s": len(want) / t, "seconds": t, "digest": dig_all,
                                      "digest_slow_prefix": dig_slow}

        calls = Calls(pairs)
        run_api(L, mi, opt, calls, min(4000, len(pairs)), 16)  # warm: the dispatcher and the lane contexts
        calls.collect(min(4000, len(pairs)))

        def arm(key, L_, mi_, opt_, n, n_threads):
            L_.mm_b200_launch_count(mi_, 1)
            t, cpu = run_api(L_, mi_, opt_, calls, n, n_threads)
            launches = L_.mm_b200_launch_count(mi_, 1)
            got = calls.collect(n)
            out["arms"][key] = {"threads": n_threads, "pairs": n, "reads": 2 * n, "reads_per_s": 2 * n / t, "seconds": t,
                                "caller_cpu_us_per_call": cpu / n * 1e6, "launches": launches, "digest": digest(got)}

        for T in [int(x) for x in args.threads.split(",")]:
            arm(f"mm_map_frag_{T}t", L, mi, opt, n_slow if T == 1 else len(pairs), T)
        L.mm_idx_destroy(mi)

        if args.parent_lib:
            P = load(args.parent_lib)
            pmi, popt = index(P, ref)
            run_api(P, pmi, popt, calls, 200, 1)  # warm
            calls.collect(200)
            for T in (1, 16):
                arm(f"parent_mm_map_frag_{T}t", P, pmi, popt, n_slow, T)
            P.mm_idx_destroy(pmi)

        for k, a in out["arms"].items():
            if k != "map_batches":
                a["digest_equal"] = a["digest"] == (dig_slow if a["pairs"] == n_slow else dig_all)
        out["all_digests_equal"] = all(a.get("digest_equal", True) for a in out["arms"].values())
        print(json.dumps(out))
    finally:
        shutil.rmtree(d, ignore_errors=True)


if __name__ == "__main__":
    main()
