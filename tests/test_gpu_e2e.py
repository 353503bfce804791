"""End-to-end parity: the B200 CLI vs the reference fork (Oracle B binary, oracle/_ref/minimap2_B, built from the
reference sources by oracle/Makefile) on the same synthetic files.
Every output line except @PG must be identical: position, strand, CIGAR, MAPQ, tags, flags.  Where the reference fork is
not built, the output is checked against its digest recorded in tests/golden/digests.json (_libs.check_digest)."""
import os
import subprocess
import pytest
import _libs as L

pytestmark = pytest.mark.gpu
NEW = os.path.join(L.ROOT, "build", "minimap2-b200")
SYN = os.path.join(L.ROOT, "build", "mmsynth")


@pytest.fixture(scope="module")
def data(tmp_path_factory):
    if not (os.path.exists(NEW) and os.path.exists(SYN)):
        pytest.skip("needs build/minimap2-b200 and build/mmsynth")
    d = tmp_path_factory.mktemp("e2e")
    subprocess.check_call([SYN, "ref", str(d / "ref.fa"), "3000000", "3", "42"])
    subprocess.check_call([SYN, "sr", str(d / "ref.fa"), str(d / "r1.fq"), str(d / "r2.fq"), "30000", "44", "0.05"])
    subprocess.check_call([SYN, "long", str(d / "ref.fa"), str(d / "long.fq"), "150", "45"])
    # edge cases the reference handles: empty read, read shorter than k, all-N read, lower case, U bases
    with open(d / "edge.fq", "w") as f:
        f.write("@short\nACGTACGT\n+\nIIIIIIII\n@allN\n" + "N" * 150 + "\n+\n" + "I" * 150 + "\n")
        ref = open(d / "ref.fa").read().split("\n")
        s = "".join(ref[1:4])[:150]
        f.write("@lower\n" + s.lower() + "\n+\n" + "I" * len(s) + "\n@rna\n" + s.replace("T", "U") + "\n+\n" + "I" * len(s) + "\n")
    return d


def _run(binary, args, cwd):
    p = subprocess.run([binary] + args, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert p.returncode == 0, p.stderr.decode()[-800:]
    return [l for l in p.stdout.decode().split("\n") if not l.startswith("@PG")]


@pytest.mark.parametrize("args", [
    ["-x", "sr", "-t", "8", "ref.fa", "r1.fq", "r2.fq"],
    ["-ax", "sr", "-t", "8", "ref.fa", "r1.fq", "r2.fq"],
    ["-ax", "sr", "-t", "3", "-K", "2M", "ref.fa", "r1.fq", "r2.fq"],       # many mini-batches
    ["-ax", "sr", "-t", "8", "ref.fa", "r1.fq"],                             # single-end through the frag path
    ["-ax", "sr", "-t", "8", "--cs", "--MD", "-Y", "ref.fa", "r1.fq", "r2.fq"],
    ["-ax", "sr", "-t", "8", "-f", "20,60", "ref.fa", "r1.fq", "r2.fq"],     # low occurrence cut-offs: re-chain path
    ["-cx", "sr", "-t", "8", "--eqx", "ref.fa", "r2.fq"],
    ["-ax", "sr", "-t", "4", "ref.fa", "edge.fq"],
    ["-x", "map-ont", "-t", "8", "ref.fa", "long.fq"],
    ["-ax", "map-ont", "-t", "8", "ref.fa", "long.fq"],
    ["-cx", "map-ont", "-t", "8", "--cs=long", "ref.fa", "long.fq"],
    # q == q2 && e == e2: the reference switches to ksw_extz2_sse (align.c:328-329); served by the extd2 kernels, see tests/test_extz2_identity.py
    ["-ax", "sr", "-t", "8", "-O", "12,12", "-E", "2,2", "ref.fa", "r1.fq", "r2.fq"],
    ["-ax", "map-ont", "-t", "8", "-O", "4,4", "-E", "2,2", "ref.fa", "long.fq"],
], ids=lambda a: " ".join(a[:-2]))
def test_cli_identical_to_reference(data, args):
    got = _run(NEW, args, data)
    if not L.have_ref_bin():
        L.check_digest("e2e " + " ".join(args), got)
        return
    want = _run(L.REF_BIN_B, args, data)
    assert len(want) == len(got)
    for i, (a, b) in enumerate(zip(want, got)):
        assert a == b, f"line {i}:\nref: {a[:300]}\nnew: {b[:300]}"
    L.record_reference_digest("e2e " + " ".join(args), want)


def test_two_mappers_from_the_first_batch(data):
    """The file driver lets its second mapper (second lane group, two mini-batches in flight) join after 16 mini-batches;
    MM2_B200_WARM_BATCHES=0 makes it join at once, so that a small input crosses the ordered hand-off many times."""
    args = ["-ax", "sr", "-t", "6", "-K", "1M", "ref.fa", "r1.fq", "r2.fq"]
    env = dict(os.environ, MM2_B200_WARM_BATCHES="0")
    p = subprocess.run([NEW] + args, cwd=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env)
    assert p.returncode == 0, p.stderr.decode()[-800:]
    got = [l for l in p.stdout.decode().split("\n") if not l.startswith("@PG")]
    if L.have_ref_bin():
        want = _run(L.REF_BIN_B, args, data)
        assert got == want
        L.record_reference_digest("e2e two mappers " + " ".join(args), want)
    else:
        L.check_digest("e2e two mappers " + " ".join(args), got)
    assert p.stderr.decode().count("mapped ") >= 8  # really many mini-batches


def test_device_post_path_equals_host_build(data):
    """The post-chaining stages compiled for the GPU (csrc/mmg_post.cu) and the host build of the same sources
    (MM2_B200_HOSTPATH=1) must print the same bytes; both are already compared with the reference above."""
    args = ["-ax", "sr", "-t", "8", "--cs", "ref.fa", "r1.fq", "r2.fq"]
    dev = _run(NEW, args, data)
    env = dict(os.environ, MM2_B200_HOSTPATH="1")
    p = subprocess.run([NEW] + args, cwd=data, stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env)
    assert p.returncode == 0, p.stderr.decode()[-800:]
    host = [l for l in p.stdout.decode().split("\n") if not l.startswith("@PG")]
    assert dev == host
    # and the library entry point for one fragment (mm_map_frag -> a batch of one) goes through the same device path
    assert len(dev) > 60000
