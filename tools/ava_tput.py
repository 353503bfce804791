"""All-vs-all read overlap throughput (-x ava-ont): reads mapped against themselves.

Builds a `mmsynth ref` genome (default 50 Mbp) and `mmsynth long` reads from it (default 50 000 reads, 10 kb mean), then
  - the CLI, `minimap2-b200 -x ava-ont -t T reads.fq reads.fq`, wall time including the index build;
  - the resident path: the index built once, then mm_b200_map_batches over the same reads (mini-batches of -K bases);
and reports reads/s and query Gbp/s for both, the host time spent on the unit name keys, and the share of seed hits the
self/dual filters dropped (path counter [7] over all planned seed hits).  Prints one JSON line; the card's name and power
limit are read in the same run.

    python tools/ava_tput.py [--genome 50000000] [--reads 50000] [--mean 10000] [--threads 16] [--out DIR]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SYN = os.path.join(ROOT, "build", "mmsynth")
CLI = os.path.join(ROOT, "build", "minimap2-b200")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        return q.stdout.strip().split("\n")[0]
    except (OSError, subprocess.TimeoutExpired):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genome", type=int, default=50_000_000)
    ap.add_argument("--reads", type=int, default=50_000)
    ap.add_argument("--mean", type=int, default=10_000)
    ap.add_argument("--threads", type=int, default=16)
    ap.add_argument("--batch", type=int, default=500_000_000, help="bases per mini-batch of the resident path (-K)")
    ap.add_argument("--out", default=None, help="directory for the generated data (default: a temporary one)")
    a = ap.parse_args()
    d = a.out or tempfile.mkdtemp(prefix="ava_tput_")
    os.makedirs(d, exist_ok=True)
    ref, fq = os.path.join(d, "ref.fa"), os.path.join(d, "reads.fq")
    subprocess.check_call([SYN, "ref", ref, str(a.genome), "8", "31"])
    subprocess.check_call([SYN, "long", ref, fq, str(a.reads), "32", str(a.mean)])
    n_bases = 0
    with open(fq, "rb") as f:
        for i, line in enumerate(f):
            if i % 4 == 1:
                n_bases += len(line) - 1
    res = {"card": card(), "reads": a.reads, "query_bases": n_bases, "threads": a.threads}

    # CLI, index build included
    t0 = time.time()
    with open(os.devnull, "wb") as null:
        subprocess.check_call([CLI, "-x", "ava-ont", "-t", str(a.threads), fq, fq], stdout=null, stderr=subprocess.DEVNULL)
    t = time.time() - t0
    res["cli"] = {"seconds": round(t, 3), "reads_per_s": round(a.reads / t, 1), "query_gbp_per_s": round(n_bases / t / 1e9, 4)}

    # resident path: index once, then the batches
    import bench
    lib = bench.load_lib()
    lib.mm_b200_name_key_time.restype = C.c_double
    lib.mm_b200_name_key_time.argtypes = [C.c_int]
    ipt, opt = bench.IdxOpt(), bench.MapOptFull()
    lib.mm_set_opt(None, C.byref(ipt), C.byref(opt))
    lib.mm_set_opt(b"ava-ont", C.byref(ipt), C.byref(opt))
    rd = lib.mm_idx_reader_open(fq.encode(), C.byref(ipt), None)
    mi = lib.mm_idx_reader_read(rd, a.threads)
    lib.mm_idx_reader_close(rd)
    lib.mm_mapopt_update(C.byref(opt), mi)
    reader = lib.mm_b200_open_reads(1, (C.c_char_p * 1)(fq.encode()))
    bs = []
    while True:
        b = lib.mm_b200_read_batch(reader, C.byref(opt), a.batch)
        if not b:
            break
        bs.append(b)
    lib.mm_b200_close_reads(reader)
    arr = (C.c_void_p * len(bs))(*bs)
    pc = (C.c_uint64 * 8)()
    for rep in range(2):  # the first pass warms the pools and the lazily made target keys
        for b in bs:
            lib.mm_b200_reset_batch(b)
        lib.mm_b200_stats(None, 1)
        lib.mm_b200_path_counts(mi, pc, 1)
        lib.mm_b200_name_key_time(1)
        t0 = time.time()
        assert lib.mm_b200_map_batches(mi, C.byref(opt), a.threads, arr, len(bs), 0) == 0
        t = time.time() - t0
    st = bench.Stats()
    lib.mm_b200_stats(C.byref(st), 0)
    lib.mm_b200_path_counts(mi, pc, 0)
    res["resident"] = {"seconds": round(t, 3), "reads_per_s": round(a.reads / t, 1), "query_gbp_per_s": round(n_bases / t / 1e9, 4),
                       "batches": len(bs), "name_key_host_s": round(lib.mm_b200_name_key_time(0), 4),
                       "seed_hits": int(st.n_anchors), "dropped_by_name": int(pc[7]),
                       "dropped_share": round(pc[7] / max(st.n_anchors, 1), 4)}
    for b in bs:
        lib.mm_b200_free_batch(b)
    lib.mm_idx_destroy(mi)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
