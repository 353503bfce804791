#!/usr/bin/env python3
"""Reads/s of airlift_b200.mappy: Aligner.map() (one call per read pair) from 1, 16 and 64 Python threads and
Aligner.map_batch(), next to the batch path (mm_b200_map_batches) on the same `mmsynth sr` pairs.  Modelled on api_tput.py.

map() goes through mm_map_frag, whose concurrent calls are mapped together as shared mini-batches (host/apiq.c); the Python
work of each call (encoding, unpacking the hits into Alignment objects) is part of what is timed, as a user pays for it.  The
one-thread arm maps the first --slow-pairs pairs only.  Every arm's hits are digested and must equal map_batch's on the same
pairs.  The card's name and power limit are read in the same run (nvidia-smi query only) and printed with the rates as one JSON
line.  Needs a GPU and build/mmsynth."""
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
from airlift_b200 import mappy  # noqa: E402
from api_tput import gpu_info, read_pairs  # noqa: E402


def digest(per_pair):
    h = hashlib.sha256()
    for i, hs in enumerate(per_pair):
        h.update(repr((i, [(a.ctg, a.r_st, a.r_en, a.strand, a.q_st, a.q_en, a.mapq, a.cigar_str, a.is_primary, a.read_num)
                           for a in hs])).encode())
    return h.hexdigest()[:16]


def run_map(al, pairs, n, n_threads):
    """map() of the first n pairs over n_threads callers; wall seconds and the hits"""
    got = [None] * n
    go = threading.Barrier(n_threads + 1)

    def work(t):
        go.wait()
        for k in range(t, n, n_threads):
            (n1, s1), (_, s2) = pairs[k]
            got[k] = list(al.map(s1, s2, name=n1))
    th = [threading.Thread(target=work, args=(t,)) for t in range(n_threads)]
    for t in th:
        t.start()
    go.wait()
    t0 = time.perf_counter()
    for t in th:
        t.join()
    return time.perf_counter() - t0, got


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genome-bp", type=int, default=100_000_000)
    ap.add_argument("--contigs", type=int, default=4)
    ap.add_argument("--pairs", type=int, default=200_000)
    ap.add_argument("--slow-pairs", type=int, default=5_000, help="pairs of the one-thread map() arm")
    ap.add_argument("--threads", default="1,16,64")
    args = ap.parse_args()
    card = gpu_info()
    bench.ensure_tools()
    cores = os.cpu_count() or 1
    d = tempfile.mkdtemp(prefix="mappy_tput_")
    try:
        ref, r1, r2 = (os.path.join(d, x) for x in ("ref.fa", "r1.fq", "r2.fq"))
        subprocess.check_call([bench.SYNTH, "ref", ref, str(args.genome_bp), str(args.contigs), "42"])
        subprocess.check_call([bench.SYNTH, "sr", ref, r1, r2, str(args.pairs), "44"])
        pairs = read_pairs(r1, r2)
        n_slow = min(args.slow_pairs, len(pairs))
        out = {"gpu": card, "cores": cores, "genome_bp": args.genome_bp, "pairs": len(pairs), "slow_pairs": n_slow, "preset": "sr",
               "arms": {}}
        L = bench.load_lib()
        L.mm_b200_set_lanes(4)
        L.mm_b200_set_in_flight(2)
        al = mappy.Aligner(ref, preset="sr")
        if not al:
            raise SystemExit("index construction failed")

        # the batch path on the files, with the aligner's index and options
        opt = bench.MapOptFull()
        C.memmove(C.byref(opt), C.byref(al._map_opt), C.sizeof(opt))
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
        for rep in range(2):  # the first pass warms every buffer to its working size
            for b in bs:
                L.mm_b200_reset_batch(b)
            t0 = time.perf_counter()
            if L.mm_b200_map_batches(al._idx, C.byref(opt), cores, arr, len(bs), 0) != 0:
                raise SystemExit("mapping failed")
            t = time.perf_counter() - t0
        for b in bs:
            L.mm_b200_free_batch(b)
        out["arms"]["mm_b200_map_batches"] = {"reads": 2 * len(pairs), "reads_per_s": 2 * len(pairs) / t, "seconds": t}

        reads = [(s1, s2) for (_, s1), (_, s2) in pairs]
        names = [n1 for (n1, _), _ in pairs]
        al.map_batch(reads[:20000], names=names[:20000])  # warm
        t0 = time.perf_counter()
        want = al.map_batch(reads, names=names)
        t = time.perf_counter() - t0
        dig_all, dig_slow = digest(want), digest(want[:n_slow])
        out["arms"]["map_batch"] = {"reads": 2 * len(pairs), "reads_per_s": 2 * len(pairs) / t, "seconds": t, "digest": dig_all}

        run_map(al, pairs, min(4000, len(pairs)), 16)  # warm: the dispatcher and the lane contexts
        for T in [int(x) for x in args.threads.split(",")]:
            n = n_slow if T == 1 else len(pairs)
            t, got = run_map(al, pairs, n, T)
            dg = digest(got)
            out["arms"][f"map_{T}t"] = {"threads": T, "pairs": n, "reads": 2 * n, "reads_per_s": 2 * n / t, "seconds": t, "digest": dg,
                                        "digest_equal": dg == (dig_slow if n == n_slow else dig_all)}
        al.close()
        out["all_digests_equal"] = all(a.get("digest_equal", True) for a in out["arms"].values())
        print(json.dumps(out))
    finally:
        shutil.rmtree(d, ignore_errors=True)


if __name__ == "__main__":
    main()
