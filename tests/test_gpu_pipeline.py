"""The place where the path plugs into AirLift: tools/airlift/0-align_reads.sh and 0-align_singletons.sh take the reference
scripts' positional arguments (src/0-align_reads.sh:3-10) and produce ${OUT_PREFIX}.bam through the same
`| samtools view -h -F4 | samtools sort` pipe (src/0-align_reads.sh:13).  samtools is not part of this image, so the test puts
a stand-in on PATH that does what those two invocations do to SAM text (drop FLAG&4 records; pass through); the records that
arrive must be the reference fork's (`minimap2_B -ax sr -R ...`) mapped records, byte for byte.
Where the reference fork is not built, those records are held to their digest recorded in tests/golden/digests.json.
Also: `--gpus 2` (reads sharded over two GPUs, index replicated) prints the same bytes as one GPU."""
import os
import stat
import subprocess
import pytest
import _libs as L

pytestmark = pytest.mark.gpu
NEW = os.path.join(L.ROOT, "build", "minimap2-b200")
SYN = os.path.join(L.ROOT, "build", "mmsynth")

FAKE_SAMTOOLS = r'''#!/usr/bin/env python3
import sys
a = sys.argv[1:]
if a and a[0] == "view":      # view -h -F4: header kept, unmapped records dropped
    for line in sys.stdin.buffer:
        if line.startswith(b"@") or not (int(line.split(b"\t", 2)[1]) & 4):
            sys.stdout.buffer.write(line)
elif a and a[0] == "sort":    # order is not what this test is about
    sys.stdout.buffer.write(sys.stdin.buffer.read())
else:
    sys.exit(2)
'''


@pytest.fixture(scope="module")
def world(tmp_path_factory):
    if not (os.path.exists(NEW) and os.path.exists(SYN)):
        pytest.skip("needs build/minimap2-b200 and build/mmsynth")
    d = tmp_path_factory.mktemp("pipe")
    subprocess.check_call([SYN, "pair", str(d / "yeast"), "12000000", "16", "42", "43", "--old"], stderr=subprocess.DEVNULL)
    subprocess.check_call([SYN, "srp", str(d / "yeast"), str(d / "reads_1.fastq"), str(d / "reads_2.fastq"), "40000", "44"])
    subprocess.check_call([SYN, "srp", str(d / "yeast"), str(d / "singletons.fastq"), str(d / "unused.fastq"), "5000", "46"])
    b = d / "bin"
    b.mkdir()
    (b / "samtools").write_text(FAKE_SAMTOOLS)
    os.chmod(b / "samtools", os.stat(b / "samtools").st_mode | stat.S_IEXEC)
    return d


def _mapped(sam_bytes):
    return [l for l in sam_bytes.split(b"\n") if l and not l.startswith(b"@PG") and (l.startswith(b"@") or not (int(l.split(b"\t", 2)[1]) & 4))]


def test_align_reads_script_is_a_drop_in(world):
    d = world
    env = dict(os.environ, PATH=str(d / "bin") + os.pathsep + os.environ["PATH"])
    rg = "@RG\\tID:S1\\tSM:S1\\tPL:illumina\\tLB:S1"
    for script, fq, ref_args in (("0-align_reads.sh", "reads", ["reads_1.fastq", "reads_2.fastq"]), ("0-align_singletons.sh", "singletons.fastq", ["singletons.fastq"])):
        out = d / ("out_" + script.split(".")[0])
        subprocess.check_call(["bash", os.path.join(L.ROOT, "tools", "airlift", script), "unused-bindir", "yeast.new.fa", fq, str(out), "8", "2", "S1", "1G"],
                              cwd=d, env=env, stderr=subprocess.DEVNULL)
        got = _mapped(open(str(out) + ".bam", "rb").read())
        assert len(got) > 1000 and any(l.startswith(b"@RG") for l in got)
        if not L.have_ref_bin():
            L.check_digest("airlift " + script, got)
            continue
        p = subprocess.run([L.REF_BIN_B, "-ax", "sr", "-R", rg, "-t", "8", "yeast.new.fa"] + ref_args, cwd=d, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
        assert p.returncode == 0
        want = _mapped(p.stdout)
        assert len(want) > 1000 and any(l.startswith(b"@RG") for l in want)
        assert got == want, script
        L.record_reference_digest("airlift " + script, want)


def test_two_gpus_print_the_same_bytes(world):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    d = world
    args = ["-ax", "sr", "-t", "8", "yeast.new.fa", "reads_1.fastq", "reads_2.fastq"]
    one = subprocess.run([NEW] + args, cwd=d, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
    two = subprocess.run([NEW, "--gpus", "2"] + args, cwd=d, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
    assert one.returncode == 0 and two.returncode == 0
    strip = lambda b: [l for l in b.split(b"\n") if not l.startswith(b"@PG")]
    assert strip(one.stdout) == strip(two.stdout) and len(strip(one.stdout)) > 80000
