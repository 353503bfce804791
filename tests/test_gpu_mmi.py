"""Index files: `-d` must write the bytes the reference writes (mm_idx_dump, index.c:438-477), and a .mmi written
by the reference must map like the FASTA it came from (mm_idx_load, index.c:479-531).  Where the reference fork is not built,
the reference's outputs are stood in for by this project's, held to their digests recorded in tests/golden/digests.json."""
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
    d = tmp_path_factory.mktemp("mmi")
    subprocess.check_call([SYN, "ref", str(d / "ref.fa"), "3000000", "3", "42"])
    subprocess.check_call([SYN, "sr", str(d / "ref.fa"), str(d / "r1.fq"), str(d / "r2.fq"), "4000", "44", "0.05"])
    subprocess.check_call([SYN, "long", str(d / "ref.fa"), str(d / "long.fq"), "40", "45"])
    return d


def _ok(cmd, cwd):
    p = subprocess.run(cmd, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert p.returncode == 0, p.stderr.decode()[-800:]
    return p


def _ref_dump(args, out, cwd):
    """the reference's `-d out` (args: index options): without the reference fork, this project's, held to the recorded digest"""
    if L.have_ref_bin():
        _ok([L.REF_BIN_B] + args + ["-d", out, "ref.fa"], cwd)
        L.record_reference_digest("mmi " + " ".join(args), open(cwd / out, "rb").read())
    else:
        _ok([NEW] + args + ["-d", out, "ref.fa"], cwd)
        L.check_digest("mmi " + " ".join(args), open(cwd / out, "rb").read())


@pytest.mark.parametrize("args", [["-x", "sr"], ["-x", "map-ont"], ["-H", "-k", "19", "-w", "10"], ["-x", "sr", "-I", "1M"],
                                  ["-k", "12", "-w", "3"]], ids=" ".join)
def test_dump_is_byte_identical(data, args):
    _ref_dump(args, "want.mmi", data)
    _ok([NEW] + args + ["-d", "got.mmi", "ref.fa"], data)
    want, got = open(data / "want.mmi", "rb").read(), open(data / "got.mmi", "rb").read()
    assert len(want) == len(got)
    if want != got:
        at = next(i for i in range(len(want)) if want[i] != got[i])
        raise AssertionError(f"first difference at byte {at} of {len(want)}")


@pytest.mark.parametrize("preset,reads", [("sr", ["r1.fq", "r2.fq"]), ("map-ont", ["long.fq"])])
def test_prebuilt_index_maps_like_fasta(data, preset, reads):
    _ref_dump(["-x", preset], f"{preset}.mmi", data)
    want = [l for l in _ok([L.REF_BIN_B if L.have_ref_bin() else NEW, "-ax", preset, "-t", "8", "ref.fa"] + reads, data).stdout.decode().split("\n")
            if not l.startswith("@PG")]
    if L.have_ref_bin():
        L.record_reference_digest(f"mmi map -ax {preset} " + " ".join(reads), want)
    else:
        L.check_digest(f"mmi map -ax {preset} " + " ".join(reads), want)
    got = [l for l in _ok([NEW, "-ax", preset, "-t", "8", f"{preset}.mmi"] + reads, data).stdout.decode().split("\n") if not l.startswith("@PG")]
    assert want == got


def test_dump_of_loaded_index_round_trips(data):
    """reading a .mmi and writing it again (-d with a .mmi input) keeps the bytes"""
    _ref_dump(["-x", "sr"], "a.mmi", data)
    _ok([NEW, "-x", "sr", "-d", "b.mmi", "a.mmi"], data)
    assert open(data / "a.mmi", "rb").read() == open(data / "b.mmi", "rb").read()
