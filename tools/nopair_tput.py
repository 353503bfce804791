#!/usr/bin/env python3
"""What --no-pairing costs: reads/s of the same human-size read pairs mapped jointly (-x sr) and with MM_F_INDEPEND_SEG
(--no-pairing), in one process and alternating the two, so that both see the same GPU, clocks and neighbours.

  resident: mm_b200_map_batches over the same parsed mini-batches (two in flight, the path bench.py times), each mode --reps times
  cli:      build/minimap2-b200 -ax sr [--no-pairing], steady state from the CLI's own log (bench.cli_mapping_phase)

Under --no-pairing every read is its own mapping unit: twice as many units, each with about half the anchors, and no pairing.
The card's name and power limit are read in the same run and printed with the rates (one JSON line on stdout).
Needs a GPU and the synthetic human-size pair that bench.py generates (tools/mmsynth.c; cached in bench.workdir())."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

MM_F_INDEPEND_SEG = 0x20000


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    if q.returncode != 0:
        raise SystemExit("nvidia-smi failed: this measurement needs a GPU")
    name, power, clk = [x.strip() for x in q.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "sm_max_clock": clk}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genome-bp", type=int, default=3_100_000_000)
    ap.add_argument("--contigs", type=int, default=24)
    ap.add_argument("--pairs", type=int, default=500_000, help="pairs per mini-batch")
    ap.add_argument("--batches", type=int, default=6, help="mini-batches per resident pass")
    ap.add_argument("--reps", type=int, default=3, help="resident passes per mode, alternating")
    ap.add_argument("--cli-pairs", type=int, default=4_000_000)
    ap.add_argument("--cli-reps", type=int, default=2)
    args = ap.parse_args()
    card = gpu_info()
    wl = bench.Workload(argparse.Namespace(workload="sr", genome_bp=args.genome_bp, contigs=args.contigs, pairs=args.pairs))
    bench.ensure_tools()
    d = bench.workdir(int(wl.G * 1.02) + 10 * (1 << 30) + (args.pairs * args.batches + args.cli_pairs) * 700)
    prefix = bench.make_pair(d, wl)
    n_res = args.pairs * (args.batches + 2)
    files = bench.make_reads(d, wl, prefix, n_res, 46, f"sr_{wl.G}_nopair_{n_res}")
    cli_files = bench.make_reads(d, wl, prefix, args.cli_pairs, 47, f"sr_{wl.G}_nopair_cli_{args.cli_pairs}")
    cores = os.cpu_count() or 1
    out = {"gpu": card, "workload": wl.config()["workload"], "cores": cores}

    # ---- CLI first, before this process holds the GPU (as bench.py does)
    cli = {"joint": [], "no_pairing": []}
    for rep in range(args.cli_reps):
        for mode in ("joint", "no_pairing"):
            det = {}
            cmd = [bench.CLI_BIN, "-ax", "sr"] + (["--no-pairing"] if mode == "no_pairing" else []) + \
                  ["-t", str(cores), "-K", str(wl.bases_per_step), prefix + ".new.fa"] + cli_files
            t = bench.cli_mapping_phase(cmd, detail=det)
            cli[mode].append({"mapping_phase_reads_per_s": 2 * args.cli_pairs / t, "steady_reads_per_s": det.get("steady")})
    out["cli"] = {"sample": f"{args.cli_pairs} pairs, build/minimap2-b200 -ax sr -t {cores} -K {wl.bases_per_step}, runs alternating", **cli}

    # ---- resident: the same parsed mini-batches through mm_b200_map_batches
    L = bench.load_lib()
    L.mm_b200_set_devices(1, (C.c_int * 1)(0))
    L.mm_b200_set_lanes(4)
    L.mm_b200_set_in_flight(2)
    ipt, opt = bench.IdxOpt(), bench.MapOptFull()
    L.mm_set_opt(None, C.byref(ipt), C.byref(opt))
    L.mm_set_opt(b"sr", C.byref(ipt), C.byref(opt))
    opt.flag |= 0x004 | 0x008
    rd = L.mm_idx_reader_open((prefix + ".new.fa").encode(), C.byref(ipt), None)
    mi = L.mm_idx_reader_read(rd, 3)
    L.mm_idx_reader_close(rd)
    if not mi:
        raise SystemExit("index construction failed")
    L.mm_mapopt_update(C.byref(opt), mi)
    nopair = bench.MapOptFull()
    C.memmove(C.byref(nopair), C.byref(opt), C.sizeof(opt))
    nopair.flag |= MM_F_INDEPEND_SEG
    fns = (C.c_char_p * 2)(*[f.encode() for f in files])
    reader = L.mm_b200_open_reads(2, fns)
    warm = [L.mm_b200_read_batch(reader, C.byref(opt), wl.bases_per_step) for _ in range(2)]
    bs = [L.mm_b200_read_batch(reader, C.byref(opt), wl.bases_per_step) for _ in range(args.batches)]
    L.mm_b200_close_reads(reader)
    if not all(warm + bs):
        raise SystemExit("ran out of synthetic reads")
    n_reads = 0
    for b in bs:
        ns = C.c_int(0)
        L.mm_b200_batch_info(b, C.byref(ns), None, None)
        n_reads += ns.value
    modes = {"joint": opt, "no_pairing": nopair}

    def run(o, batches):
        arr = (C.c_void_p * len(batches))(*batches)
        t0 = time.perf_counter()
        if L.mm_b200_map_batches(mi, C.byref(o), cores, arr, len(batches), 0) != 0:
            raise SystemExit("mapping failed")
        t = time.perf_counter() - t0  # the call returns with every hit on the host
        nh = C.c_int64(0)
        dig = sum(L.mm_b200_batch_digest(b, C.byref(nh)) for b in batches) & (2**64 - 1)
        for b in batches:
            L.mm_b200_reset_batch(b)
        return t, dig

    for o in modes.values():  # every buffer at its working size for both unit layouts
        run(o, warm + bs[:2])
    res = {m: [] for m in modes}
    digests = {m: set() for m in modes}
    for rep in range(args.reps):
        for m, o in modes.items():
            t, dig = run(o, bs)
            res[m].append(n_reads / t)
            digests[m].add(dig)
    out["resident"] = {"sample": f"{args.batches} mini-batches of {args.pairs} pairs ({n_reads} reads), mm_b200_map_batches, two in flight, "
                                 f"{args.reps} passes per mode alternating",
                       **{m: {"reads_per_s": v, "median": sorted(v)[len(v) // 2]} for m, v in res.items()},
                       "same_hits_every_pass": all(len(v) == 1 for v in digests.values()),
                       "modes_differ": digests["joint"] != digests["no_pairing"]}
    for b in warm + bs:
        L.mm_b200_free_batch(b)
    L.mm_idx_destroy(mi)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
