"""All-vs-all modes on the GPU (-D, -X, --dual=no, -x ava-ont): the self/dual filters of skip_seed (map.c:125-147) on the
device, held to the strcmp oracle (tests/aux/ava_oracle.c) anchor for anchor and chain for chain, and the CLI held to
identities that need no reference build."""
import ctypes as C
import hashlib
import os
import subprocess
import numpy as np
import pytest
import _libs as L
import _ava as A
from test_gpu_no_pairing import Api

pytestmark = pytest.mark.gpu
SYN = os.path.join(L.ROOT, "build", "mmsynth")
NEW = os.path.join(L.ROOT, "build", "minimap2-b200")
GOLD = os.path.join(L.ROOT, "tests", "golden", "cli")
MM_F_CIGAR, MM_F_OUT_SAM = 0x004, 0x008

# size and sha256 of the ava-ont outputs of test_cli_ava_ont: this project's own output on a B200, recorded where no reference
# build was available.  They guard against regressions; they do not prove parity with the reference.
CLI_DIGESTS = {
    "-x ava-ont reads.fq reads.fq":
        {"bytes": 8553137, "sha256": "7a1b1a5193dd6f29d275d4434b3cd0f463148c96f446d16834838e41bcae53c2"},
    "-cx ava-ont reads.fq reads.fq":
        {"bytes": 166281077, "sha256": "366670aed52106d40ceeafe290861988e3cd5712f98f82152ec700cc84a949dc"},
}


@pytest.fixture(scope="module")
def gpu():
    import airlift_b200.api as api
    ctx = api.Context(0)
    rng = np.random.default_rng(5)
    names, seqs = A.make_targets(rng)
    idx = api.Index(ctx, seqs, A.W, A.K)
    idx.set_names(names)
    T = A.Targets(names, seqs)
    yield api, ctx, idx, T, A.make_queries(rng, names, seqs)
    T.close()
    idx.close()
    ctx.close()


@pytest.mark.parametrize("heap", [0, 1], ids=["radix", "heap"])
def test_anchors_equal_strcmp_oracle(gpu, heap):
    api, ctx, idx, T, queries = gpu
    n_self = 0
    for qname, q in queries:
        mv, qlen = L.frag_minimizers(L.orc_sketch, [q], A.W, A.K)
        for flag in A.FLAGS + [0]:
            flag |= A.MM_F_HEAP_SORT if heap else 0
            want, rep, _ = T.collect(qname, heap, flag, 1000, mv, qlen)
            got, rep2, _ = ctx.collect_seeds(idx, heap, flag, 1000, mv, qlen, len(mv) * 8 + 64, name=qname)
            assert got.tobytes() == want.tobytes() and rep2 == rep, (qname, hex(flag))
            n_self += int(((want["y"] & A.SEED_SELF) != 0).sum())
    assert n_self > 0


def _oracle_chains(T, qname, q, opt):
    """mm_map_frag up to chaining (map.c:295-377) with the strcmp oracle, the max_occ re-chain included; also the hits the
    self/dual filters dropped in the passes taken"""
    O = A.oracle_named()
    mv, qlen = L.frag_minimizers(L.orc_sketch, [q], A.W, A.K)
    heap = bool(opt.flag & A.MM_F_HEAP_SORT)
    params = (opt.max_gap, opt.max_gap, opt.bw, opt.max_chain_skip, opt.max_chain_iter, opt.min_cnt, opt.min_chain_score, 0, 1)
    a, rep, nn = T.collect(qname, heap, opt.flag, opt.mid_occ, mv, qlen)
    u, b = L.chain_call(O.orc_chain_dp, params, a)
    if opt.max_occ > opt.mid_occ and rep > 0 and len(u) == 0:  # one segment: re-chained only when nothing chained (map.c:353-375)
        a, rep, nn2 = T.collect(qname, heap, opt.flag, opt.max_occ, mv, qlen)
        u, b = L.chain_call(O.orc_chain_dp, params, a)
        nn += nn2
    return u, b, nn


@pytest.mark.parametrize("mode", ["radix", "heap", "rechain"])
def test_batch_chains_equal_oracle(gpu, mode):
    api, ctx, idx, T, queries = gpu
    for flag in (A.MM_F_NO_DIAG, A.MM_F_NO_DUAL, A.MM_F_NO_DIAG | A.MM_F_NO_DUAL | A.MM_F_FOR_ONLY):
        opt = api.ont_opt(1000)
        opt.flag |= flag | (A.MM_F_HEAP_SORT if mode != "radix" else 0)
        if mode == "rechain":  # -f x,y: a low first cut-off, re-chained with the higher one
            opt.mid_occ, opt.max_occ = 1, 1000
        frags = [[q] for _, q in queries] * 3
        names = [n for n, _ in queries] * 3
        batch, keep = api.Context.make_batch(frags)
        ctx.path_counts(reset=True)
        ctx.batch_upload(opt, batch, names=names, idx=idx)
        ch = api.chains_to_py(ctx.seed_chain_resident(idx, opt, True))
        n_named = 0
        for f, (qname, q) in enumerate(zip(names, [x[0] for x in frags])):
            u, b, nn = _oracle_chains(T, qname, q, opt)
            uo, ao = int(ch["u_off"][f]), int(ch["a_off"][f])
            assert ch["n_u"][f] == len(u) and (ch["u"][uo:uo + len(u)] == u).all(), (f, qname, hex(opt.flag))
            assert ch["a"][ao:ao + len(b)].tobytes() == b.tobytes(), (f, qname, hex(opt.flag))
            n_named += nn
        pc = ctx.path_counts()
        assert int(pc[7]) == n_named and n_named > 0
        if mode == "rechain":
            assert int(ch["rechained"].sum()) > 0


def test_flips_and_names_in_one_upload(gpu):
    """a flip table and unit keys in one upload: the queries uploaded reverse-complemented, every flip set, chain exactly as the
    queries as read, both under their names, and the name filters drop the same hits"""
    api, ctx, idx, T, queries = gpu
    opt = api.ont_opt(1000)
    opt.flag |= A.MM_F_NO_DIAG | A.MM_F_NO_DUAL | A.MM_F_HEAP_SORT
    names = [n for n, _ in queries]
    runs = []
    for frags, flips in (([[q] for _, q in queries], None), ([[L.revcomp(q)] for _, q in queries], np.ones(len(queries), np.uint8))):
        batch, keep = api.Context.make_batch(frags)
        ctx.path_counts(reset=True)
        ctx.batch_upload(opt, batch, flips=flips, names=names, idx=idx)
        runs.append((api.chains_to_py(ctx.seed_chain_resident(idx, opt, True)), int(ctx.path_counts()[7])))
    (want, want_named), (got, got_named) = runs
    for k in ("n_u", "n_a", "rep_len", "n_mini", "rechained", "u_off", "a_off", "mini_off"):
        assert np.array_equal(got[k], want[k]), k
    assert got["u"].tobytes() == want["u"].tobytes() and got["a"].tobytes() == want["a"].tobytes()
    assert np.array_equal(got["mini_pos"], want["mini_pos"])
    assert got_named == want_named > 0 and int(want["n_u"].sum()) > 0


def test_missing_name_keys_refused(gpu):
    api, ctx, idx, T, queries = gpu
    opt = api.ont_opt(1000)
    opt.flag |= A.MM_F_NO_DUAL
    batch, keep = api.Context.make_batch([[q] for _, q in queries])
    ctx.batch_upload(opt, batch)  # no unit keys for this batch
    with pytest.raises(api.MmgError, match=r"mmg_batch_t\.ukey"):
        ctx.seed_chain_resident(idx, opt, True)
    bare = api.Index(ctx, T.seqs, A.W, A.K)  # no target keys
    try:
        ctx.batch_upload(opt, batch, names=[n for n, _ in queries], idx=idx)
        with pytest.raises(api.MmgError, match="mmg_idx_set_name_keys"):
            ctx.seed_chain_resident(bare, opt, True)
    finally:
        bare.close()
    ctx.batch_upload(opt, batch, names=[n for n, _ in queries], idx=idx)
    ctx.batch_upload(opt, batch)  # a new upload drops the keys of the batch before
    with pytest.raises(api.MmgError):
        ctx.seed_chain_resident(idx, opt, True)


# ---------------------------------------------------------------------------------------------------- CLI

def _run(args, cwd):
    p = subprocess.run([NEW] + args, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert p.returncode == 0, p.stderr.decode()[-800:]
    return [l for l in p.stdout.decode().split("\n") if l and not l.startswith("@PG")]


def _renamed_ref(src, dst, prefix):
    import gzip
    with gzip.open(src, "rb") as f, open(dst, "wb") as o:
        for line in f:
            o.write(b">" + prefix + line[1:] if line.startswith(b">") else line)


@pytest.fixture(scope="module")
def longfix(tmp_path_factory):
    if not os.path.exists(NEW):
        pytest.skip("needs build/minimap2-b200")
    d = tmp_path_factory.mktemp("ava_long")
    _renamed_ref(os.path.join(GOLD, "ref.fa.gz"), d / "ref.fa", b"")
    _renamed_ref(os.path.join(GOLD, "ref.fa.gz"), d / "after.fa", b"~")   # '~' sorts after every read name
    _renamed_ref(os.path.join(GOLD, "ref.fa.gz"), d / "before.fa", b"!")  # '!' sorts before
    subprocess.check_call(["sh", "-c", f"gzip -dc {GOLD}/long.fq.gz > {d}/long.fq"])
    return d


@pytest.mark.parametrize("fmt", [["-c"], ["-a"]], ids=["paf", "sam"])
def test_cli_filters_that_change_nothing(longfix, fmt):
    base = _run(fmt + ["-x", "map-ont", "-t", "8", "ref.fa", "long.fq"], longfix)
    assert len([l for l in base if not l.startswith("@")]) >= 8
    assert _run(fmt + ["-x", "map-ont", "-D", "-t", "8", "ref.fa", "long.fq"], longfix) == base  # no read is named like a target
    after = _run(fmt + ["-x", "map-ont", "-t", "8", "after.fa", "long.fq"], longfix)
    assert _run(fmt + ["-x", "map-ont", "--dual=no", "-t", "8", "after.fa", "long.fq"], longfix) == after
    before = _run(fmt + ["-x", "map-ont", "--dual=no", "-t", "8", "before.fa", "long.fq"], longfix)
    if fmt == ["-c"]:
        assert before == []
    else:
        recs = [l for l in before if not l.startswith("@")]
        assert len(recs) > 0 and all(int(l.split("\t")[1]) & 0x4 for l in recs)


@pytest.fixture(scope="module")
def overlap(tmp_path_factory):
    if not (os.path.exists(SYN) and os.path.exists(NEW)):
        pytest.skip("needs build/mmsynth and build/minimap2-b200")
    d = tmp_path_factory.mktemp("ava")
    subprocess.check_call([SYN, "ref", str(d / "ref.fa"), "2000000", "2", "17"])
    subprocess.check_call([SYN, "long", str(d / "ref.fa"), str(d / "reads.fq"), "4000", "18", "10000"])
    return d


def _paf_ok(lines):
    n = 0
    for l in lines:
        f = l.split("\t")
        assert f[0].encode() <= f[5].encode(), l[:200]                             # --dual=no: each pair once
        assert not (f[0] == f[5] and f[2] == f[7] and f[3] == f[8] and f[4] == "+"), l[:200]  # -D: no diagonal self-hit
        n += 1
    return n


def _digest(key, lines):
    blob = "\n".join(lines).encode()
    got = {"bytes": len(blob), "sha256": hashlib.sha256(blob).hexdigest()}
    assert CLI_DIGESTS.get(key) == got, f"{key!r}: {got}"


@pytest.mark.parametrize("x", ["-x", "-cx"])
def test_cli_ava_ont(overlap, x):
    args = [x, "ava-ont", "reads.fq", "reads.fq"]
    one = _run(["-t", "8"] + args, overlap)
    assert _paf_ok(one) > 4000
    assert _run(["-t", "1"] + args, overlap) == one
    # mm_map_frag, read by read under its own name, gives the records of the CLI (keys follow the shards and the batches)
    api = Api(overlap / "reads.fq", b"ava-ont")
    try:
        opt = api.opt_with(0)
        opt.flag &= ~(MM_F_OUT_SAM | (0 if x == "-cx" else MM_F_CIGAR))
        by = {}
        for l in one:
            f = l.split("\t")
            by.setdefault(f[0], []).append((f[5], int(f[7]), int(f[8]), int(f[2]), int(f[3]), int(f[4] == "-"), int(f[11])))
        fq = open(overlap / "reads.fq", "rb").read().split(b"\n")
        names = [fq[i][1:].split()[0] for i in range(0, len(fq) - 3, 4)]
        seqs = [fq[i + 1] for i in range(0, len(fq) - 3, 4)]
        checked = 0
        for k in range(0, len(names), 10):
            hits, _ = api.map_frag(names[k], [seqs[k]], opt)
            got = [(names[h[0]].decode(), h[1], h[2], h[3], h[4], h[5], h[6]) for h in hits[0]]
            assert got == by.get(names[k].decode(), []), names[k]
            checked += len(got)
        assert checked > 100
    finally:
        api.close()
    _digest(" ".join(args), one)


def test_cli_ava_two_gpus(overlap):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    args = ["-x", "ava-ont", "-t", "8", "reads.fq", "reads.fq"]
    assert _run(["--gpus", "2"] + args, overlap) == _run(["--gpus", "1"] + args, overlap)
