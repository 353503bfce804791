#!/usr/bin/env python3
"""Index load times: build from FASTA, load a .mmi with sequences, load a .mmi written with --idx-no-seq.

The reference is the `mmsynth pair` reference bench.py maps against (3.1 Gbp, 24 contigs, seeds 42/43), or with --small a
100 Mbp one.  The two .mmi files are written by build/minimap2-b200 -d (not timed).  Each load is timed in this process around
mm_idx_reader_read, which returns once the device index is complete, after one untimed load that initialises CUDA.  Prints
one JSON line: wall seconds per run of each load, mmg_idx_bytes (HBM footprint) of each index, and the GPU it ran on.
Everything is written under --dir (default: a new temporary directory)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = os.path.join(ROOT, "build", "minimap2-b200")
SYN = os.path.join(ROOT, "build", "mmsynth")
LIB = os.path.join(ROOT, "airlift_b200", "libmm2b200.so")


def _lib():
    lib = C.CDLL(LIB)
    P = C.c_void_p
    for f, res, args in [("mm_idx_reader_open", P, [C.c_char_p, P, C.c_char_p]), ("mm_idx_reader_read", P, [P, C.c_int]),
                         ("mm_idx_reader_close", None, [P]), ("mm_idx_destroy", None, [P]), ("mm_b200_didx", P, [P, C.c_int]),
                         ("mmg_idx_bytes", C.c_size_t, [P]), ("mmg_device_count", C.c_int, []), ("mm_set_opt", C.c_int, [C.c_char_p, P, P])]:
        getattr(lib, f).restype = res
        getattr(lib, f).argtypes = args
    return lib


def load(lib, fn, preset):
    """(seconds, mmg_idx_bytes) of reading the first index part of fn with the preset's index options"""
    io, mo = C.create_string_buffer(256), C.create_string_buffer(1024)  # mm_idxopt_t, mm_mapopt_t
    lib.mm_set_opt(None, io, mo)
    lib.mm_set_opt(preset.encode(), io, mo)
    t0 = time.perf_counter()
    rd = lib.mm_idx_reader_open(os.fsencode(fn), io, None)
    mi = lib.mm_idx_reader_read(rd, 8)
    dt = time.perf_counter() - t0
    lib.mm_idx_reader_close(rd)
    if not mi:
        raise SystemExit(f"cannot load {fn}")
    nbytes = lib.mmg_idx_bytes(lib.mm_b200_didx(mi, 0))
    lib.mm_idx_destroy(mi)
    return dt, nbytes


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--small", action="store_true", help="a 100 Mbp reference instead of the 3.1 Gbp one")
    ap.add_argument("--preset", default="sr")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--dir", default=None)
    a = ap.parse_args()
    lib = _lib()
    if lib.mmg_device_count() < 1:
        raise SystemExit("no CUDA device: nothing to measure")
    d = a.dir or tempfile.mkdtemp(prefix="mmi_noseq_")
    bp, n_ctg = (100_000_000, 4) if a.small else (3_100_000_000, 24)
    prefix = os.path.join(d, "pair")
    if not os.path.exists(prefix + ".new.fa"):
        subprocess.check_call([SYN, "pair", prefix, str(bp), str(n_ctg), "42", "43"])
    fa, seq_mmi, noseq_mmi = prefix + ".new.fa", os.path.join(d, "seq.mmi"), os.path.join(d, "noseq.mmi")
    if not os.path.exists(seq_mmi):
        subprocess.check_call([NEW, "-x", a.preset, "-v", "1", "-d", seq_mmi, fa])
    if not os.path.exists(noseq_mmi):
        subprocess.check_call([NEW, "-x", a.preset, "-v", "1", "--idx-no-seq", "-d", noseq_mmi, fa])
    load(lib, noseq_mmi, a.preset)  # CUDA initialisation, page cache
    res = {"fasta": [], "mmi": [], "mmi_noseq": []}
    size = {}
    for _ in range(a.runs):  # the three loads alternate, so that drift hits all alike
        for k, fn in (("fasta", fa), ("mmi", seq_mmi), ("mmi_noseq", noseq_mmi)):
            t, size[k] = load(lib, fn, a.preset)
            res[k].append(round(t, 3))
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         stderr=subprocess.DEVNULL, text=True).stdout.strip().splitlines()
    print(json.dumps({"reference_bp": bp, "preset": a.preset, "runs": a.runs, "load_s": res, "idx_bytes": size,
                      "file_bytes": {"mmi": os.path.getsize(seq_mmi), "mmi_noseq": os.path.getsize(noseq_mmi)},
                      "gpu": gpu[0] if gpu else None}))


if __name__ == "__main__":
    main()
