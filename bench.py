#!/usr/bin/env python
"""bench.py -- reads/s of the re-alignment hot path on N B200s (one process per GPU).

Workload (BASELINE.json configs[2] / [4], the one `north_star` names): a human-size synthetic reference pair
(3.1 Gbp, 24 contigs, repeat families, N runs, hg19->hg38-shaped edits; tools/mmsynth.c `pair`, seeds 42/43) and 2x150 bp FR
pairs drawn from its updated / retired regions (read seed 44 + rank), mapped with the `-ax sr` preset against the NEW
reference.  One step = one mini-batch of pairs through the whole hot path (sketch -> seed -> chain -> hits -> ksw2 extension
-> MAPQ/pairing), i.e. worker_pipeline's step 1 of the reference (map.c:590-593).  `--workload ont` runs configs[3]
(10 kb ONT-shaped reads overlapping the same updated regions, `-ax map-ont`); `--genome-bp`/`--contigs` give configs[0]/[1].

  value    : reads/s with the batch already resident in HBM (mm_b200_map_batch mode 2)
  e2e      : reads/s through the batch C-ABI with HOST buffers (mode 0: H2D of the reads, all stages, D2H of the hit
             records, malloc'd mm_reg1_t out) -- the same scope the reference arm times
  cli      : the whole drop-in binary (FASTQ parse + map + SAM), next to the reference CLI on the same files
  parity   : before anything is timed, a prefix of the workload is mapped through the same in-process index and its SAM
             records are compared byte for byte with the reference fork's (oracle/_ref/minimap2_B); at N>1 every rank
             maps the same prefix with its replica of the index and the digests must agree
  roofline : the dominant kernel by CUDA-event time inside the timed region
  --dump-outputs DIR : the hits of the last mini-batch of the resident timed pass, one float64 array per field (dump_outputs), so
             that two builds can be compared hit for hit on the same seeded inputs
  --impl reference / cpu_baseline : the reference fork's own mapping step (worker_pipeline step 1 = kt_for(worker_for) ->
             mm_map_frag, unmodified objects in oracle/_ref/libmm2ref.so driven by oracle/ref_mapstep.c) on all host
             cores, same files, same mini-batch size; parsing and SAM formatting run but are not in the step time
             (they are in `cli`).
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
LIB = os.path.join(ROOT, "airlift_b200", "libmm2b200.so")
SYNTH = os.path.join(ROOT, "build", "mmsynth")
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "minimap2_B")
REF_STEP = os.path.join(ROOT, "oracle", "_ref", "ref_mapstep")
CLI_BIN = os.path.join(ROOT, "build", "minimap2-b200")
TRAFFIC_JSON = os.path.join(ROOT, "profiles", "traffic_r02.json")   # dram bytes per launch from the committed ncu --set full captures
# integer-pipe roofline of K4 (SURVEY.md 8d): 148 SMs x 128 lanes x 1.965 GHz lane-ops/s over ~30 lane-ops per DP cell (one cell per lane-op)
K4_INT_ROOFLINE_GCUPS = 148 * 128 * 1.965 / 30.0

METRIC = "remapped reads/sec at 1/2/4/8 B200; ksw2 GCUPS; seed-lookup HBM GB/s"
PARITY_PAIRS = 100_000
# --dump-outputs: the columns of mm_b200_batch_hits (include/minimap_b200.h), and the size cap of all files together (npy headers aside)
HIT_FIELDS = ("read", "rid", "rs", "re", "qs", "qe", "rev", "mapq", "score", "primary", "sam_pri", "proper_frag", "mlen", "blen",
              "dp_score", "dp_max", "n_cigar")
DUMP_BYTES = (64 << 20) - (1 << 16)
# (workload, genome bp, contigs, parity units) -> (records, sha256) of oracle/_ref/minimap2_B's SAM records of the parity prefix,
# from runs where the reference fork was built (profiles/bench_r02_n1.json, "reference_sha256"): without it the gate compares with these
REF_PARITY = {("sr", 3_100_000_000, 24, PARITY_PAIRS): (200_000, "18d83c22c05360e9b758914f3a2637e4e1b1ede46a93dbd87c2d5ca13616f2a2")}


class IdxOpt(C.Structure):
    _fields_ = [("k", C.c_short), ("w", C.c_short), ("flag", C.c_short), ("bucket_bits", C.c_short), ("mini_batch_size", C.c_int),
                ("batch_size", C.c_uint64)]


class MapOptFull(C.Structure):  # mm_mapopt_t (include/minimap_b200.h == minimap.h:107-150)
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


class Stats(C.Structure):  # mm_b200_stats_t
    _fields_ = [(n, C.c_double) for n in ("t_total", "t_upload", "t_seedchain", "t_seedchain_kernels", "t_hits", "t_align_host",
                                          "t_ksw_total", "t_ksw_kernel", "t_finish")] + \
               [(n, C.c_uint64) for n in ("n_frag", "n_reads", "n_bases", "n_minimizers", "n_anchors", "n_chain_iter", "n_dp_jobs",
                                          "n_dp_cells", "n_dp_rounds", "h2d_bytes", "d2h_bytes", "n_dp_jobs_fast", "n_dp_cells_fast")]


def load_lib():
    if not os.path.exists(LIB):
        raise SystemExit(f"{LIB} missing: run `make` (the CUDA library is the product; there is no CPU fallback)")
    from airlift_b200.dist import IdxImage
    L = C.CDLL(LIB)
    L.mm_set_opt.argtypes = [C.c_char_p, C.POINTER(IdxOpt), C.POINTER(MapOptFull)]
    L.mm_idx_reader_open.restype = C.c_void_p
    L.mm_idx_reader_open.argtypes = [C.c_char_p, C.POINTER(IdxOpt), C.c_char_p]
    L.mm_idx_reader_read.restype = C.c_void_p
    L.mm_idx_reader_read.argtypes = [C.c_void_p, C.c_int]
    L.mm_idx_reader_close.argtypes = [C.c_void_p]
    L.mm_idx_destroy.argtypes = [C.c_void_p]
    L.mm_mapopt_update.argtypes = [C.POINTER(MapOptFull), C.c_void_p]
    L.mm_b200_set_devices.argtypes = [C.c_int, C.POINTER(C.c_int)]
    L.mm_b200_open_reads.restype = C.c_void_p
    L.mm_b200_open_reads.argtypes = [C.c_int, C.POINTER(C.c_char_p)]
    L.mm_b200_close_reads.argtypes = [C.c_void_p]
    L.mm_b200_read_batch.restype = C.c_void_p
    L.mm_b200_read_batch.argtypes = [C.c_void_p, C.POINTER(MapOptFull), C.c_int]
    L.mm_b200_batch_info.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int64)]
    L.mm_b200_map_batch.argtypes = [C.c_void_p, C.POINTER(MapOptFull), C.c_int, C.c_void_p, C.c_int]
    L.mm_b200_map_batches.argtypes = [C.c_void_p, C.POINTER(MapOptFull), C.c_int, C.POINTER(C.c_void_p), C.c_int, C.c_int]
    L.mm_b200_batches_in_flight.argtypes = [C.c_void_p, C.POINTER(MapOptFull)]
    L.mm_b200_reset_batch.argtypes = [C.c_void_p]
    L.mm_b200_free_batch.argtypes = [C.c_void_p]
    L.mm_b200_write_batch.argtypes = [C.c_void_p, C.POINTER(MapOptFull), C.c_void_p]
    L.mm_b200_batch_digest.restype = C.c_uint64
    L.mm_b200_batch_digest.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
    L.mm_b200_batch_hits.restype = C.c_int64
    L.mm_b200_batch_hits.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]
    L.mm_b200_stats.argtypes = [C.POINTER(Stats), C.c_int]
    L.mm_b200_profile.argtypes = [C.c_void_p, C.c_int]
    L.mm_b200_set_serial.argtypes = [C.c_int]
    L.mm_b200_profile_fetch.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_double), C.POINTER(C.c_long)]
    L.mm_b200_idx_image.argtypes = [C.c_void_p, C.c_void_p]
    L.mm_b200_idx_alloc_named.restype = C.c_void_p
    L.mm_b200_idx_alloc_named.argtypes = [C.POINTER(IdxOpt), C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_uint32), C.POINTER(IdxImage), C.POINTER(IdxImage)]
    L.mm_b200_idx_seq.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_uint32)]
    L.mm_b200_idx_finalize.argtypes = [C.c_void_p]
    L.mmg_memcpy_d2d.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    L.mm_b200_ctx.restype = C.c_void_p
    L.mm_b200_ctx.argtypes = [C.c_void_p, C.c_int]
    L.mmg_stream.restype = C.c_void_p
    L.mmg_stream.argtypes = [C.c_void_p]
    L.mm_b200_path_counts.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.c_int]
    L.mmg_growth_counts.argtypes = [C.POINTER(C.c_uint64), C.c_int]
    L.mm_b200_launch_count.restype = C.c_long
    L.mm_b200_launch_count.argtypes = [C.c_void_p, C.c_int]
    return L


def ensure_tools():
    if not os.path.exists(SYNTH):
        subprocess.check_call(["make", "-C", ROOT, "tools"], stdout=subprocess.DEVNULL)


def workdir(need_bytes=0):
    """/dev/shm when it can hold the synthetic files of all ranks (what is already there from an earlier run counts), else the
    temp dir.  Every rank evaluates this before anything is written, so all ranks pick the same place."""
    import shutil
    for base in (["/dev/shm"] if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else []) + [tempfile.gettempdir()]:
        d = os.path.join(base, "airlift_b200_bench")
        have = sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) if os.path.isdir(d) else 0
        if base != "/dev/shm" or shutil.disk_usage(base).free + have >= need_bytes * 1.1 + (1 << 30):
            os.makedirs(d, exist_ok=True)
            return d


class Workload:
    """names, presets and sizes of one BASELINE.json config"""

    def __init__(self, args):
        self.kind = args.workload
        self.G, self.n_ctg = args.genome_bp, args.contigs
        self.size_name = ("Human-size" if self.G >= 2_000_000_000 else "C. elegans-size" if self.G >= 50_000_000 else "Yeast-size")
        if self.kind == "sr":
            self.preset, self.k, self.w = "sr", 21, 11
            self.units = args.pairs or 500_000                   # pairs per step
            self.reads_per_unit, self.bases_per_step = 2, (args.pairs or 500_000) * 300
        else:
            self.preset, self.k, self.w = "map-ont", 15, 10
            self.units = args.pairs or 10_000                    # long reads per step
            self.reads_per_unit, self.bases_per_step = 1, (args.pairs or 10_000) * 10_000
        self.prefix_name = f"pair_{self.G}_{self.n_ctg}"

    def config(self):
        if self.kind == "sr":
            what = f"2x150bp reads from updated/retired regions, minimap2 -ax sr; {self.units} pairs per step"
        else:
            what = f"10 kb ONT-shaped reads overlapping updated regions, minimap2 -ax map-ont; {self.units} reads per step"
        return {"workload": f"{self.size_name} synthetic pair ({self.G / 1e6:.0f} Mbp, {self.n_ctg} contigs, hg19->hg38-shaped edits), {what}",
                "preset": self.preset, "k": self.k, "w": self.w, "units_per_step": self.units, "mini_batch_bases": self.bases_per_step,
                "shards": "one job sharded by reads: every rank maps reads drawn (read seed 44 + rank) from the same updated regions (edit seed 43)",
                "l2_policy": "inputs larger than L2 (the index alone is >20 GB at human size; 150 MB of reads per step), a different batch every step"}


def make_pair(d, wl):
    """the reference pair: <prefix>.new.fa / .regions.bed / .src.fa (tools/mmsynth.c pair, ref seed 42, edit seed 43)"""
    prefix = os.path.join(d, wl.prefix_name)
    if not os.path.exists(prefix + ".ok"):
        tmp = prefix + f".tmp{os.getpid()}"
        subprocess.check_call([SYNTH, "pair", tmp, str(wl.G), str(wl.n_ctg), "42", "43"])
        for ext in (".new.fa", ".regions.bed", ".src.fa"):
            os.replace(tmp + ext, prefix + ext)
        open(prefix + ".ok", "w").write("ok\n")
    return prefix


def make_reads(d, wl, prefix, n_units, read_seed, tag):
    if wl.kind == "sr":
        f1, f2 = os.path.join(d, f"{tag}_1.fq"), os.path.join(d, f"{tag}_2.fq")
        if not (os.path.exists(f1) and os.path.exists(f2)):
            t1, t2 = f1 + f".tmp{os.getpid()}", f2 + f".tmp{os.getpid()}"
            subprocess.check_call([SYNTH, "srp", prefix, t1, t2, str(n_units), str(read_seed)])
            os.replace(t1, f1)
            os.replace(t2, f2)
        return [f1, f2]
    f1 = os.path.join(d, f"{tag}.fq")
    if not os.path.exists(f1):
        t1 = f1 + f".tmp{os.getpid()}"
        subprocess.check_call([SYNTH, "long", prefix + ".new.fa", t1, str(n_units), str(read_seed), "10000", prefix + ".regions.bed"])
        os.replace(t1, f1)
    return [f1]


def ref_index(d, wl, prefix, cores):
    """the reference fork's own index of the new reference (`minimap2_B -d`), built once per box and kept next to the FASTA"""
    mmi = f"{prefix}.{wl.preset}.ref.mmi"
    secs = None
    if not os.path.exists(mmi):
        tmp = mmi + f".tmp{os.getpid()}"
        t0 = time.time()
        subprocess.check_call([REF_BIN, "-x", wl.preset, "-t", str(cores), "-d", tmp, prefix + ".new.fa"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        os.replace(tmp, mmi)
        secs = time.time() - t0
    return mmi, secs


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.samples, self.reasons, self.max_mhz, self._halt = gpu_index, [], set(), None, threading.Event()

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def cli_mapping_phase(cmd, out_path=None, detail=None):
    """Run a minimap2-style CLI; return seconds between `loaded/built the index` and `Real time` (BASELINE.md section 3).
    detail (a dict) receives `steady`: reads/s between the second and the last `mapped N sequences` line of the CLI's own log,
    i.e. without the start-up of the first two mini-batches (buffer growth, pipeline fill)."""
    out = open(out_path, "wb") if out_path else subprocess.DEVNULL
    p = subprocess.run(cmd, stdout=out, stderr=subprocess.PIPE, text=True)
    if out_path:
        out.close()
    t_idx = t_end = None
    done = []
    for line in p.stderr.splitlines():
        m = re.match(r"\[M::main::([0-9.]+)\*", line)
        if m and "loaded/built the index" in line:
            t_idx = float(m.group(1))
        m = re.match(r"\[M::worker_pipeline::([0-9.]+)\*[0-9.]+\] mapped (\d+) sequences", line)
        if m:
            done.append((float(m.group(1)), int(m.group(2))))
        m = re.search(r"Real time: ([0-9.]+) sec", line)
        if m:
            t_end = float(m.group(1))
    if p.returncode != 0 or t_idx is None or t_end is None:
        raise RuntimeError("CLI run failed: " + p.stderr[-400:])
    if detail is not None and len(done) >= 4 and done[-1][0] > done[1][0]:
        detail["steady"] = sum(n for _, n in done[2:]) / (done[-1][0] - done[1][0])
        detail["steady_sample"] = f"mini-batches 3..{len(done)} by the CLI's own log timestamps"
    return t_end - t_idx


def ref_mapstep(mmi, files, wl, cores, n_batches):
    """the reference fork's worker_pipeline, step 1 timed alone (oracle/ref_mapstep.c)"""
    cmd = [REF_STEP, "-x", wl.preset, "-a", "-t", str(cores), "-K", str(wl.bases_per_step), "-n", str(n_batches), mmi] + files
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    if p.returncode != 0:
        raise RuntimeError("ref_mapstep failed: " + p.stderr[-400:])
    return json.loads(p.stdout.strip().splitlines()[-1])


def run_reference(args, wl, d):
    """--impl reference: the reference fork's mapping step on the host cores, same files and mini-batch size as the repo arm."""
    if not (os.path.exists(REF_BIN) and os.path.exists(REF_STEP)):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/{minimap2_B,ref_mapstep} are not built (make -C oracle ref needs /root/reference)"}))
        return
    cores = os.cpu_count() or 1
    prefix = make_pair(d, wl)
    n_steps = args.warmup + args.steps
    files = make_reads(d, wl, prefix, wl.units * n_steps, 44, f"{wl.kind}_{wl.G}_r44_{wl.units}x{n_steps}")
    mmi, idx_s = ref_index(d, wl, prefix, cores)
    r = ref_mapstep(mmi, files, wl, cores, n_steps)
    if r["batches"] < n_steps:
        raise SystemExit(f"reference arm: {r['batches']} mini-batches read, {n_steps} expected")
    ms = r["map_s"][args.warmup:]
    reads = sum(r["reads"][args.warmup:])
    per_step = sum(ms) / len(ms)
    v = reads / sum(ms)
    # the whole reference CLI (parse + map + SAM, its 3-stage pipeline overlapping) on the same files, for the `cli` comparison
    cli = None
    if not args.no_cli:
        try:
            det = {}
            t = cli_mapping_phase([REF_BIN, "-ax", wl.preset, "-t", str(cores), "-K", str(wl.bases_per_step), mmi] + files, detail=det)
            cli = {"value": sum(r["reads"]) / t, "unit": "reads/s", "sample": f"{sum(r['reads'])} reads in {n_steps} mini-batches, minimap2_B -ax {wl.preset} -t {cores} -K {wl.bases_per_step}, "
                   "mapping phase (index loaded) incl. FASTQ parsing and SAM output", "steady_state": det.get("steady"), "steady_state_sample": det.get("steady_sample")}
        except Exception as e:  # noqa
            cli = {"value": None, "unit": "reads/s", "sample": f"failed: {e}"}
    sample = (f"{args.steps} timed mini-batches of {wl.units} {'pairs' if wl.kind == 'sr' else 'reads'} after {args.warmup} warm-up ones, the reference's own step 1 "
              f"(kt_for(worker_for) -> mm_map_frag, map.c:590-593) on {cores} threads; parsing and SAM formatting run outside the step time")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "reads/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/int32",
        "data": "synthetic", "config": wl.config(),
        "cpu_baseline": {"value": v, "unit": "reads/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "cli": cli, "index": {"file": os.path.basename(mmi), "build_s": idx_s, "load_s": r["index_s"], "mid_occ": r["mid_occ"]},
        "host_s_per_step": {"parse": sum(r["read_s"]) / n_steps, "map": per_step, "format": sum(r["write_s"]) / n_steps}}))


def sam_records(path):
    """(count, sha256) of the non-header lines of a SAM/PAF file"""
    h, n = hashlib.sha256(), 0
    with open(path, "rb") as f:
        for line in f:
            if not line.startswith(b"@"):
                h.update(line)
                n += 1
    return n, h.hexdigest()


def first_difference(p1, p2):
    with open(p1, "rb") as a, open(p2, "rb") as b:
        la = (l for l in a if not l.startswith(b"@"))
        lb = (l for l in b if not l.startswith(b"@"))
        for i, (x, y) in enumerate(zip(la, lb)):
            if x != y:
                return i, x[:200].decode(errors="replace"), y[:200].decode(errors="replace")
    return None


def batch_hits(L, b):
    """the hits of a mapped batch as its caller receives them: (rows of HIT_FIELDS in read order, their CIGAR words concatenated)"""
    import numpy as np
    n_cig = C.c_int64(0)
    n = L.mm_b200_batch_hits(b, None, None, C.byref(n_cig))
    rows = np.zeros((n, len(HIT_FIELDS)), dtype=np.int64)
    cig = np.zeros(n_cig.value, dtype=np.uint32)
    L.mm_b200_batch_hits(b, rows.ctypes.data, cig.ctypes.data, C.byref(n_cig))
    return rows, cig


def dump_outputs(out_dir, rows, cig, n_reads):
    """Writes out_dir/<field>.npy (one float64 per hit, fields of HIT_FIELDS) and out_dir/cigar.npy (the CIGAR words of those hits in
    hit order; n_cigar.npy splits them).  Over DUMP_BYTES, whole reads are kept in a fixed seeded order until the budget is spent,
    so that equal hits give equal files.  Returns (hits written, reads kept)."""
    import numpy as np
    n_cigar = rows[:, HIT_FIELDS.index("n_cigar")]
    hit_bytes = 8 * (len(HIT_FIELDS) + n_cigar)
    read_bytes = np.bincount(rows[:, 0], weights=hit_bytes, minlength=n_reads)
    order = np.random.default_rng(0).permutation(n_reads)
    keep_read = np.zeros(n_reads, dtype=bool)
    keep_read[order[np.cumsum(read_bytes[order]) <= DUMP_BYTES]] = True
    keep = keep_read[rows[:, 0]]
    os.makedirs(out_dir, exist_ok=True)
    for j, name in enumerate(HIT_FIELDS):
        np.save(os.path.join(out_dir, f"{name}.npy"), rows[keep, j].astype(np.float64))
    np.save(os.path.join(out_dir, "cigar.npy"), cig[np.repeat(keep, n_cigar)].astype(np.float64))
    return int(keep.sum()), int(keep_read.sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="sr", choices=["sr", "ont"])
    ap.add_argument("--genome-bp", type=int, default=3_100_000_000)
    ap.add_argument("--contigs", type=int, default=24)
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--pairs", type=int, default=0, help="pairs (sr) or reads (ont) per step; default 500000 / 10000")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the SAM-identity gate against oracle/_ref/minimap2_B")
    ap.add_argument("--no-long-read", action="store_true", help="skip the map-ont run appended to the short-read line at N=1")
    ap.add_argument("--no-cli", action="store_true", help="skip the whole-CLI (parse + map + SAM) timing at N=1")
    ap.add_argument("--lanes", type=int, default=4, help="streams per GPU: two mini-batches in flight, each cut into lanes/2 shards")
    ap.add_argument("--in-flight", type=int, default=2, help="mini-batches in flight (each on lanes/in_flight streams)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the hits of the last timed mini-batch to DIR/<field>.npy (float64); --impl b200 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the b200 path computes; --impl reference has no such outputs")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    wl = Workload(args)

    ensure_tools()
    n_steps = max(args.warmup, 4) + args.steps * (2 if os.environ.get("BENCH_E2E_TWICE") else 1)   # the b200 arm warms up on at least four mini-batches
    bytes_per_unit = 700 if wl.kind == "sr" else 20_500
    d = workdir(int(wl.G * 1.02) + 10 * (1 << 30) + world * wl.units * n_steps * bytes_per_unit)
    if args.impl == "reference":
        if rank == 0:
            run_reference(args, wl, d)
        return

    cores = os.cpu_count() or 1
    have_ref = os.path.exists(REF_BIN) and os.path.exists(REF_STEP)
    t_setup0 = time.time()
    if rank == 0:
        prefix = make_pair(d, wl)

    cli_result = None
    if rank == 0 and world == 1 and not args.no_cli and os.path.exists(CLI_BIN):
        # the whole drop-in binary (FASTQ parse + all stages + SAM on stdout), timed exactly like the reference CLI; it runs
        # before this process touches the GPU, so that the binary sees the device a user's run would see
        n_units = wl.units * 8
        cf = make_reads(d, wl, prefix, n_units, 45, f"{wl.kind}_{wl.G}_cli_{n_units}")
        try:
            det = {}
            t = cli_mapping_phase([CLI_BIN, "-ax", wl.preset, "-t", str(cores), "-K", str(wl.bases_per_step), prefix + ".new.fa"] + cf, detail=det)
            cli_result = {"value": wl.reads_per_unit * n_units / t, "unit": "reads/s", "steady_state": det.get("steady"), "steady_state_sample": det.get("steady_sample"),
                          "sample": f"{n_units} {'pairs' if wl.kind == 'sr' else 'reads'} in 8 mini-batches, build/minimap2-b200 -ax {wl.preset} -t {cores} -K {wl.bases_per_step}, "
                                    "mapping phase (after the index is built) incl. FASTQ parsing, first-batch buffer growth and SAM output"}
        except Exception as e:  # noqa
            cli_result = {"value": None, "unit": "reads/s", "sample": f"failed: {e}"}

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()  # the pair exists from here on
    prefix = os.path.join(d, wl.prefix_name)
    # one job, sharded: every rank maps reads of the same updated regions (SURVEY.md 8d); rank r draws its own reads
    read_seed = 44 + rank
    files = make_reads(d, wl, prefix, wl.units * n_steps, read_seed, f"{wl.kind}_{wl.G}_r{read_seed}_{wl.units}x{n_steps}")
    par_units = PARITY_PAIRS if wl.kind == "sr" else 1000
    par_files = None
    if not args.no_parity:
        if rank == 0:
            par_files = make_reads(d, wl, prefix, par_units, 4400, f"{wl.kind}_{wl.G}_parity_{par_units}")
        if world > 1:
            dist.barrier()
        par_files = make_reads(d, wl, prefix, par_units, 4400, f"{wl.kind}_{wl.G}_parity_{par_units}")
    t_data = time.time() - t_setup0

    L = load_lib()
    libc = C.CDLL(None)
    dev = (C.c_int * 1)(local_rank)
    L.mm_b200_set_devices(1, dev)
    L.mm_b200_set_lanes(args.lanes)
    L.mm_b200_set_in_flight(args.in_flight)
    ipt, opt = IdxOpt(), MapOptFull()
    L.mm_set_opt(None, C.byref(ipt), C.byref(opt))
    L.mm_set_opt(wl.preset.encode(), C.byref(ipt), C.byref(opt))
    opt.flag |= 0x004 | 0x008  # -a: MM_F_CIGAR | MM_F_OUT_SAM
    t0 = time.time()
    bcast_bytes = 0
    if world == 1 or rank == 0:
        rd = L.mm_idx_reader_open((prefix + ".new.fa").encode(), C.byref(ipt), None)
        mi = L.mm_idx_reader_read(rd, 3)
        L.mm_idx_reader_close(rd)
        if not mi:
            raise SystemExit("index construction failed")
        L.mm_mapopt_update(C.byref(opt), mi)
    t_build = time.time() - t0
    if world > 1:
        # the index is built once (rank 0) and replicated: one NCCL broadcast per buffer over NVLink/NVSwitch;
        # nothing else is ever exchanged between ranks
        from airlift_b200 import dist as D
        img = D.IdxImage()
        names = None
        if rank == 0:
            assert L.mm_b200_idx_image(mi, C.byref(img)) == 0
            names = []
            for i in range(img.n_seq):
                nm, ln = C.c_char_p(), C.c_uint32()
                L.mm_b200_idx_seq(mi, i, C.byref(nm), C.byref(ln))
                names.append((nm.value, ln.value))
        shape = D.broadcast_object((img.shape_tuple(), opt.mid_occ, names) if rank == 0 else None)
        if rank != 0:
            shp = D.IdxImage.from_shape(shape[0])
            img = D.IdxImage()
            nm_arr = (C.c_char_p * len(shape[2]))(*[x[0] for x in shape[2]])
            ln_arr = (C.c_uint32 * len(shape[2]))(*[x[1] for x in shape[2]])
            mi = L.mm_b200_idx_alloc_named(C.byref(ipt), len(shape[2]), nm_arr, ln_arr, C.byref(shp), C.byref(img))
            opt.mid_occ = shape[1]
        bcast_bytes = D.broadcast_buffers(L, img, torch.device("cuda", local_rank), src=0)
        if rank != 0:
            L.mm_b200_idx_finalize(mi)
        torch.cuda.synchronize()
    t_index = time.time() - t0
    n_threads = args.threads or max(1, cores // world)
    ctx = L.mm_b200_ctx(mi, 0)
    stream = torch.cuda.ExternalStream(L.mmg_stream(ctx), device=torch.device("cuda", local_rank))

    def open_reader(fl):
        fns = (C.c_char_p * len(fl))(*[f.encode() for f in fl])
        return L.mm_b200_open_reads(len(fl), fns)

    # ---- parity gate: the SAM records of a prefix of the workload, through this very index, against the reference fork
    parity = {"ok": None, "checked": False, "why": "skipped (--no-parity)"}
    if not args.no_parity:
        rdr = open_reader(par_files)
        pb = L.mm_b200_read_batch(rdr, C.byref(opt), 2_000_000_000)
        if not pb or L.mm_b200_map_batch(mi, C.byref(opt), n_threads, pb, 0) != 0:
            raise SystemExit("parity gate: mapping failed")
        nh = C.c_int64(0)
        digest = L.mm_b200_batch_digest(pb, C.byref(nh))
        ranks_equal = None
        if world > 1:
            t = torch.tensor([digest & 0x7fffffffffffffff, nh.value], device="cuda", dtype=torch.int64)
            allv = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(allv, t)
            ranks_equal = all(bool(torch.equal(v, allv[0])) for v in allv)
        if rank == 0:
            ours = os.path.join(d, f"parity_b200_{os.getpid()}.sam")
            sys.stdout.flush()
            libc.fflush(None)
            saved = os.dup(1)
            fd = os.open(ours, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o644)
            os.dup2(fd, 1)
            try:
                L.mm_b200_write_batch(mi, C.byref(opt), pb)   # formats, prints and frees the batch
                libc.fflush(None)
            finally:
                os.dup2(saved, 1)
                os.close(fd)
                os.close(saved)
            n_ours, h_ours = sam_records(ours)
            parity = {"checked": False, "ok": None, "units": par_units, "records": n_ours, "sha256": h_ours, "hits": nh.value,
                      "ranks_digest_equal": ranks_equal, "why": "oracle/_ref/minimap2_B not built: records hashed, not compared"}
            if have_ref:
                mmi, idx_s = ref_index(d, wl, prefix, cores)
                theirs = os.path.join(d, f"parity_ref_{os.getpid()}.sam")
                cli_mapping_phase([REF_BIN, "-ax", wl.preset, "-t", str(cores), mmi] + par_files, out_path=theirs)
                n_ref, h_ref = sam_records(theirs)
                ok = (n_ref == n_ours and h_ref == h_ours and ranks_equal is not False)
                parity.update({"checked": True, "ok": ok, "reference_records": n_ref, "reference_sha256": h_ref, "reference_index_build_s": idx_s,
                               "why": "every SAM record of the prefix identical to oracle/_ref/minimap2_B's" if ok else "MISMATCH"})
                if not ok:
                    parity["first_difference"] = first_difference(ours, theirs)
                    sys.stderr.write(f"[bench] PARITY MISMATCH: {parity}\n")
                os.unlink(theirs)
            elif (wl.kind, wl.G, wl.n_ctg, par_units) in REF_PARITY:
                n_ref, h_ref = REF_PARITY[(wl.kind, wl.G, wl.n_ctg, par_units)]
                ok = (n_ref == n_ours and h_ref == h_ours and ranks_equal is not False)
                parity.update({"checked": True, "ok": ok, "reference_records": n_ref, "reference_sha256": h_ref,
                               "why": "every SAM record of the prefix identical to minimap2_B's, by its stored digest (REF_PARITY)" if ok else "MISMATCH"})
                if not ok:
                    sys.stderr.write(f"[bench] PARITY MISMATCH: {parity}\n")
            os.unlink(ours)
        else:
            L.mm_b200_free_batch(pb)
        L.mm_b200_close_reads(rdr)

    reader = open_reader(files)

    def next_batch():
        b = L.mm_b200_read_batch(reader, C.byref(opt), wl.bases_per_step)
        if not b:
            raise SystemExit("ran out of synthetic reads")
        return b

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- warm-up (full path, host buffers)
    # (through the same two-in-flight call as the timed passes, so that every lane's arenas reach their working size here)
    wb = [next_batch() for _ in range(max(args.warmup, 4))]   # at least two per lane group: both staging slots of every stream get used
    # the K mini-batches of the timed passes: parsed once, mapped three times (host buffers; resident; kernel profile).  They are
    # parsed BEFORE the warm-up, so that the timed region starts right behind it: two seconds of FASTQ parsing in between let
    # the GPU fall back to its idle clocks, and the ramp back up cost the first timed pass 30-50 ms per step.
    batches = [next_batch() for _ in range(args.steps)]
    n_reads = 0
    for b in batches:
        ns = C.c_int(0)
        L.mm_b200_batch_info(b, C.byref(ns), None, None)
        n_reads += ns.value
    for rep in range(2):
        if L.mm_b200_map_batches(mi, C.byref(opt), n_threads, (C.c_void_p * len(wb))(*wb), len(wb), 0) != 0:
            raise SystemExit("mapping failed")
        for b in wb:
            L.mm_b200_reset_batch(b)
        wb = wb[1:] + wb[:1]   # the other lane group sees the other batches
    for b in wb:
        L.mm_b200_free_batch(b)

    def timed(mode_resident, in_flight=1, profile=False, capture=False):
        """K steps; returns (seconds max over ranks, reads of all ranks, stats, kernel profile, launches, clocks, digest).
        in_flight: mini-batches resident at a time in the resident pass (1 when the shards take turns on the device).
        capture: keep the hits of the last step in timed.last_hits (rows, cigar, reads of that step)."""
        L.mm_b200_stats(None, 1)
        L.mmg_growth_counts((C.c_uint64 * 2)(), 1)
        L.mm_b200_path_counts(mi, (C.c_uint64 * 8)(), 1)
        L.mm_b200_launch_count(mi, 1)
        L.mm_b200_profile(mi, 1 if profile else 0)   # CUDA events around every launch: only in the separate profile pass
        sampler = ClockSampler(local_rank)
        sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dev_ms = 0.0
        sync_all()
        arr = (C.c_void_p * len(batches))(*batches)
        if not mode_resident:
            # the K mini-batches through the batch C-ABI, two in flight (mm_b200_map_batches): host buffers in, malloc'd hits out
            ev0.record(stream)
            if L.mm_b200_map_batches(mi, C.byref(opt), n_threads, arr, len(batches), 0) != 0:
                raise SystemExit("mapping failed")
            ev1.record(stream)
            sync_all()
            dev_ms = ev0.elapsed_time(ev1)
        else:
            # the reads of up to two mini-batches (one per lane group) are staged in HBM outside the timed region, then the resident
            # pass of those batches is timed
            for i in range(0, len(batches), in_flight):
                pair = (C.c_void_p * len(batches[i:i + in_flight]))(*batches[i:i + in_flight])
                if L.mm_b200_map_batches(mi, C.byref(opt), n_threads, pair, len(pair), 1) != 0:
                    raise SystemExit("upload failed")
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                if L.mm_b200_map_batches(mi, C.byref(opt), n_threads, pair, len(pair), 2) != 0:
                    raise SystemExit("mapping failed")
                e1.record(stream)
                torch.cuda.synchronize()
                dev_ms += e0.elapsed_time(e1)
            sync_all()
        clocks = sampler.stop()
        st = Stats()
        L.mm_b200_stats(C.byref(st), 0)
        names, ms, ln = (C.c_char_p * 64)(), (C.c_double * 64)(), (C.c_long * 64)()
        nk = L.mm_b200_profile_fetch(mi, 64, names, ms, ln)
        prof = {}
        for i in range(nk):  # template instantiations (k_ksw<16>, k_ksw<32>) count as one kernel
            nm = names[i].decode().split("<")[0]
            prof[nm] = (prof.get(nm, (0.0, 0))[0] + ms[i], prof.get(nm, (0.0, 0))[1] + ln[i])
        L.mm_b200_profile(mi, 0)
        launches = L.mm_b200_launch_count(mi, 0)
        gr = (C.c_uint64 * 2)()
        L.mmg_growth_counts(gr, 0)
        timed.growths = [int(gr[0]), int(gr[1])]
        pc = (C.c_uint64 * 8)()
        L.mm_b200_path_counts(mi, pc, 0)
        timed.paths = {"rechained": pc[0], "heap_rank_replay": pc[1], "heap_literal_replay": pc[2], "warp_tree": pc[3], "zdrop_rounds": pc[4],
                       "zdrop_cuts": pc[5], "replayed_hits": pc[6]}
        if capture:   # before the reset below drops the hits
            ns = C.c_int(0)
            L.mm_b200_batch_info(batches[-1], C.byref(ns), None, None)
            timed.last_hits = batch_hits(L, batches[-1]) + (ns.value,)
        digest = 0
        for b in batches:  # the three passes must produce the same hits
            digest ^= L.mm_b200_batch_digest(b, None)
            L.mm_b200_reset_batch(b)
        secs = dev_ms * 1e-3
        if world > 1:
            t = torch.tensor([secs, float(n_reads)], device="cuda", dtype=torch.float64)
            tmax = t.clone()
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            tsum = t.clone()
            dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
            per_rank = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(per_rank, t)
            timed.per_rank_ms = [float(x[0]) * 1e3 / args.steps for x in per_rank]
            secs, total_reads = float(tmax[0]), float(tsum[1])
        else:
            total_reads = float(n_reads)
            timed.per_rank_ms = [secs * 1e3 / args.steps]
        return secs, total_reads, st, prof, launches, clocks, digest

    secs_e2e, reads_e2e, st_e2e, prof_e2e, launches_e2e, clocks_e2e, dig_e2e = timed(False)
    growths_e2e = timed.growths
    if os.environ.get("BENCH_E2E_TWICE"):   # diagnostic: the same batches again, every arena at its final size
        r2 = timed(False)
        s2 = r2[0]
        keep = batches
        batches = [next_batch() for _ in range(args.steps)]   # a second set of new batches
        r3 = timed(False)
        sys.stderr.write(f"[bench] e2e pass 3 (other new batches) {r3[0] * 1e3 / args.steps:.1f} ms/step\n")
        for b in batches:
            L.mm_b200_free_batch(b)
        batches = keep
        for nm, st in (("pass 1", st_e2e), ("pass 2", r2[2])):
            sys.stderr.write(f"[bench] {nm}: total {st.t_total:.3f} upload {st.t_upload:.3f} seed/chain {st.t_seedchain:.3f} (kernels {st.t_seedchain_kernels:.3f}) dp {st.t_ksw_total:.3f} (kernel {st.t_ksw_kernel:.3f}) finish {st.t_finish:.3f}\n")
        sys.stderr.write(f"[bench] e2e pass 1 {secs_e2e * 1e3 / args.steps:.1f} ms/step (buffer re-allocations {growths_e2e}), pass 2 {s2 * 1e3 / args.steps:.1f} ms/step ({timed.growths})\n")
    in_flight = L.mm_b200_batches_in_flight(mi, C.byref(opt))   # 1 for the presets whose post-chaining stages run on the host
    secs_res, reads_res, st_res, prof_val, launches_res, clocks_res, dig_res = timed(True, in_flight=in_flight, capture=bool(args.dump_outputs))
    per_rank_ms = timed.per_rank_ms
    # Kernel profile: a third pass in which the shards of a GPU take turns on the device.  In the timed passes the two shards'
    # kernels overlap on purpose, which stretches every per-kernel CUDA-event interval; the roofline figures need clean ones.
    L.mm_b200_set_serial(1)
    _, _, st_res, prof_res, _, _, dig_prof = timed(True, in_flight=1, profile=True)
    L.mm_b200_set_serial(0)
    for b in batches:
        L.mm_b200_free_batch(b)

    out = None
    if rank == 0:
        peaks = {}
        pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pk):
            peaks = json.load(open(pk))
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
        # dominant kernel by device time in the resident timed region
        dom = max(prof_res.items(), key=lambda kv: kv[1][0]) if prof_res else ("none", (0.0, 0))
        dname, (dms, dn) = dom
        step_dev_ms = sum(v[0] for v in prof_res.values())
        # algorithmic HBM bytes of each kernel over the timed region (DESIGN.md section 4: bytes per unit x units from the live counters)
        nmv, nanch, cells, jobs = st_res.n_minimizers, st_res.n_anchors, st_res.n_dp_cells, st_res.n_dp_jobs
        cells_fast, jobs_fast = st_res.n_dp_cells_fast, st_res.n_dp_jobs_fast
        paths = timed.paths
        algo = {
            # serial merge replay: a rank in, a slot out per replayed hit (latency-bound: one dependent pop after the other)
            "k_heap_replay": paths["replayed_hits"] * 8.0,
            "k_sketch_count": st_res.n_bases * 0.5, "k_sketch_fill": st_res.n_bases * 0.5 + nmv * 16, "k_sketch_reads": st_res.n_bases * 0.5 + nmv * 16,
            "k_lookup": nmv * (16 + 16 + 12), "k_fill": nmv * 28 + nanch * (8 + 16), "k_expand": nmv * 28 + nanch * (8 + 16),
            "k_chain_fill": nanch * (16 + 16), "k_chain_tail_warp": nanch * (16 + 16 + 16 + 16),
            "k_ksw": (cells - cells_fast) * 1.0 + (jobs - jobs_fast) * 64, "k_ksw_dpx": (cells - cells_fast) * 1.0 + (jobs - jobs_fast) * 64,
            "k_ksw_dpx_block": (cells - cells_fast) * 1.0 + (jobs - jobs_fast) * 64, "k_ksw_tpj": cells_fast * 1.0 + jobs_fast * 64,
            "k_ksw_wave": cells_fast * 1.0 + jobs_fast * 64,
            "k_encode_reads": st_res.n_bases * 1.5,
            # post-chaining bookkeeping: chained anchors in, query + target windows as 4-bit codes, hits out
            "k_post_hits": nanch * 16 + st_res.n_bases * 1.0 + st_res.n_reads * 96, "k_post_align": cells * 0.0 + jobs * 64 + st_res.n_bases * 1.0 + st_res.n_reads * 160,
        }
        a_bytes = algo.get(dname, 0.0)
        achieved = a_bytes / (dms * 1e-3) / 1e9 if dms > 0 else 0.0
        traffic = None
        if os.path.exists(TRAFFIC_JSON):
            traffic = json.load(open(TRAFFIC_JSON)).get(dname, {}).get("dram_bytes_per_launch")
        roof = {"bound": "hbm", "kernel": dname, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "traffic": traffic, "peak_source": peak_src, "launches": dn, "avg_launch_ms": dms / dn if dn else None,
                "algorithmic_bytes_per_launch": a_bytes / dn if dn else None,
                "share_of_kernel_time": dms / step_dev_ms if step_dev_ms else None,
                "note": "the chaining and DP kernels are integer/latency-bound, not HBM-bound: their HBM fraction is small by construction; "
                        "see k4 (GCUPS against the integer-pipe roofline) and DESIGN.md section 4"}
        ksw_lit_ms = prof_res.get("k_ksw", (0.0, 0))[0] + prof_res.get("k_ksw_dpx", (0.0, 0))[0] + prof_res.get("k_ksw_dpx_block", (0.0, 0))[0]
        ksw_fast_ms = prof_res.get("k_ksw_tpj", (0.0, 0))[0] + prof_res.get("k_ksw_wave", (0.0, 0))[0]
        ksw_ms = ksw_lit_ms + ksw_fast_ms
        lookup_ms = prof_res.get("k_lookup", (0.0, 0))[0]
        gc = lambda c, ms: c / (ms * 1e-3) / 1e9 if ms else None
        k4 = {"gcups": gc(cells, ksw_ms), "gcups_fast_form": gc(cells_fast, ksw_fast_ms), "gcups_literal_form": gc(cells - cells_fast, ksw_lit_ms),
              "cells_per_step": cells / args.steps, "fast_form_cell_share": cells_fast / cells if cells else None,
              "int_roofline_gcups": K4_INT_ROOFLINE_GCUPS, "frac": (gc(cells, ksw_ms) or 0.0) / K4_INT_ROOFLINE_GCUPS,
              "roofline_def": "148 SMs x 128 int lanes x 1.965 GHz / 30 lane-ops per cell (SURVEY.md 8d, one cell per lane-op)"}
        out = {
            "metric": METRIC, "value": reads_res / secs_res, "unit": "reads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": secs_res * 1e3 / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/int32", "data": "synthetic", "config": wl.config(),
            "e2e": {"value": reads_e2e / secs_e2e, "unit": "reads/s", "h2d_bytes_per_step": st_e2e.h2d_bytes // args.steps,
                    "d2h_bytes_per_step": st_e2e.d2h_bytes // args.steps, "ms_per_step": secs_e2e * 1e3 / args.steps},
            "gpu_launches": int(launches_res), "roofline": roof, "parity": parity,
            "passes_digest_equal": bool(dig_e2e == dig_res == dig_prof), "passes_digest": [f"{x:016x}" for x in (dig_e2e, dig_res, dig_prof)],
            "ksw_gcups": k4["gcups"], "k4": k4,
            "seed_lookup_gbs": algo["k_lookup"] / (lookup_ms * 1e-3) / 1e9 if lookup_ms else None,
            "kernel_ms_per_step": {k: v[0] / args.steps for k, v in sorted(prof_res.items(), key=lambda kv: -kv[1][0])},
            "kernel_launches_per_step": {k: v[1] / args.steps for k, v in sorted(prof_res.items(), key=lambda kv: -kv[1][0])},
            "kernel_profile": "CUDA events around every launch in a separate pass of the same K steps with the two shards of a GPU serialised "
                              "(in the timed passes their kernels overlap, which stretches per-kernel intervals)",
            "paths_per_step": {k: v / args.steps for k, v in paths.items()},
            "work_per_step": {"reads": n_reads / args.steps, "bases": st_res.n_bases / args.steps, "minimizers": nmv / args.steps, "anchors": nanch / args.steps,
                              "chain_iterations": st_res.n_chain_iter / args.steps, "dp_jobs": jobs / args.steps, "dp_cells": cells / args.steps},
            "host_s_per_step": {"seed_chain_call": st_res.t_seedchain / args.steps, "hits": st_res.t_hits / args.steps,
                                "align_host": st_res.t_align_host / args.steps, "dp_call": st_res.t_ksw_total / args.steps,
                                "finish": st_res.t_finish / args.steps, "dp_rounds": st_res.n_dp_rounds / args.steps},
            "host_s_per_step_e2e": {"upload": st_e2e.t_upload / args.steps, "seed_chain_call": st_e2e.t_seedchain / args.steps, "hits": st_e2e.t_hits / args.steps,
                                    "align_host": st_e2e.t_align_host / args.steps, "dp_call": st_e2e.t_ksw_total / args.steps, "finish": st_e2e.t_finish / args.steps,
                                    "total": st_e2e.t_total / args.steps},
            "per_rank_ms_per_step": per_rank_ms, "host_threads": n_threads, "host_cores": cores,
            "setup_s": {"synthetic_data": t_data, "index_build": t_build, "index_build_and_broadcast": t_index},
            "index_broadcast_bytes": bcast_bytes, "clocks": clocks_res, "lanes": args.lanes, "batches_in_flight": in_flight, "buffer_reallocations_in_e2e_pass": {"device": growths_e2e[0], "pinned": growths_e2e[1]},
            "hbm_used_gb": (lambda fr_to: (fr_to[1] - fr_to[0]) / 1e9)(torch.cuda.mem_get_info()),
        }
    # ---- CPU baseline next to it (rank 0, N=1 only): the reference fork's mapping step on a bounded sample of the same files
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline and have_ref:
            try:
                mmi, idx_s = ref_index(d, wl, prefix, cores)
                nb = min(n_steps, 3)
                r = ref_mapstep(mmi, files, wl, cores, nb)
                ms, rd = r["map_s"][1:], r["reads"][1:]   # the first mini-batch warms the page cache and the allocator
                out["cpu_baseline"] = {"value": sum(rd) / sum(ms), "unit": "reads/s", "cores": cores, "kind": "reference",
                                       "sample": f"mini-batches 2..{nb} of the same files ({sum(rd)} reads), the reference's own step 1 (mm_map_frag on {cores} threads), "
                                                 "parsing and SAM formatting outside the step time"}
            except Exception as e:  # noqa
                out["cpu_baseline"] = {"value": None, "unit": "reads/s", "cores": cores, "kind": "reference", "sample": f"failed: {e}"}
        else:
            out["cpu_baseline"] = {"value": None, "unit": "reads/s", "cores": cores, "kind": "reference",
                                   "sample": "measured at N=1 only" if world > 1 else "skipped or oracle/_ref not built"}
        if cli_result is not None:
            out["cli"] = cli_result
    L.mm_b200_close_reads(reader)
    L.mm_idx_destroy(mi)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0 and world == 1 and wl.kind == "sr" and not args.no_long_read:
        # BASELINE.json configs[3] next to the headline: 10 kb ONT-shaped reads overlapping the same updated regions, -ax map-ont, in a
        # process of its own (another index: k=15, w=10) now that this one has released the GPU
        try:
            cmd = [sys.executable, os.path.abspath(__file__), "--workload", "ont", "--steps", "3", "--warmup", "3", "--no-cli", "--no-parity",
                   "--no-cpu-baseline", "--no-long-read", "--genome-bp", str(args.genome_bp), "--contigs", str(args.contigs)]
            p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
            lr = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
            out["long_read"] = {"workload": lr["config"]["workload"], "value": lr["value"], "unit": lr["unit"], "ms_per_step": lr["ms_per_step"],
                                "e2e": lr["e2e"], "ksw_gcups": lr["ksw_gcups"], "passes_digest_equal": lr["passes_digest_equal"],
                                "kernel_ms_per_step": dict(list(lr["kernel_ms_per_step"].items())[:6]),
                                "note": "post-chaining stages of the long-read presets run on the host (DESIGN.md section 1); parity of this preset is held by "
                                        "tests/test_gpu_e2e.py, tests/test_gpu_paths.py and the golden CLI cases"}
        except Exception as e:  # noqa
            out["long_read"] = {"value": None, "why": f"failed: {e}"}
    if rank == 0 and args.dump_outputs:
        rows, cig, n_last = timed.last_hits
        n_kept, reads_kept = dump_outputs(args.dump_outputs, rows, cig, n_last)
        out["dump_outputs"] = {"dir": args.dump_outputs, "reads": n_last, "hits": len(rows), "reads_written": reads_kept, "hits_written": n_kept}
    if rank == 0:
        print(json.dumps(out))


if __name__ == "__main__":
    main()
