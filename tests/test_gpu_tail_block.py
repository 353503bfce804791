"""The CTA form of the chain tail (k_chain_tail_block) normally takes the few fragments with thousands of anchors.
MMG_TAIL_HEAVY_N=0 sends every fragment of the first pass through it, so the chaining parity tests (oracle, golden vectors,
CLI byte identity incl. the repeat-family fixture) all run on its level-by-level backtracking; MMG_TAIL_WALK=1 selects the
chain-walking form it replaced, which stays as the path for presets with min_cnt < 2.  Both variables are read once per
process, hence the subprocesses.
The CTA form launches with more than 48 KB of shared memory, a kernel attribute every device needs: with `--gpus 2` and
MMG_TAIL_HEAVY_N=0 the second GPU's fragments all take it too, and the output must be what one GPU prints."""
import os
import subprocess
import sys
import pytest
import _libs as L

pytestmark = pytest.mark.gpu
NEW = os.path.join(L.ROOT, "build", "minimap2-b200")
SYN = os.path.join(L.ROOT, "build", "mmsynth")
SUITE = ["tests/test_gpu_kernels.py", "tests/test_golden.py", "tests/test_gpu_paths.py", "tests/test_gpu_e2e.py"]


@pytest.mark.parametrize("walk", [0, 1])
def test_chaining_suite_through_the_cta_tail(walk):
    env = dict(os.environ, MMG_TAIL_HEAVY_N="0")
    if walk:
        env["MMG_TAIL_WALK"] = "1"
    r = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", "-k", "chain or golden or paths or e2e or cli"] + SUITE,
                       cwd=L.ROOT, env=env, capture_output=True, text=True, timeout=2400)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-1000:])
    assert " passed" in r.stdout


def test_two_gpus_through_the_cta_tail(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    if not (os.path.exists(NEW) and os.path.exists(SYN)):
        pytest.skip("needs build/minimap2-b200 and build/mmsynth")
    subprocess.check_call([SYN, "ref", str(tmp_path / "ref.fa"), "3000000", "3", "42"])
    subprocess.check_call([SYN, "sr", str(tmp_path / "ref.fa"), str(tmp_path / "r1.fq"), str(tmp_path / "r2.fq"), "30000", "44", "0.05"])
    env = dict(os.environ, MMG_TAIL_HEAVY_N="0")
    out = {}
    for gpus in ("1", "2"):
        p = subprocess.run([NEW, "--gpus", gpus, "-ax", "sr", "-t", "8", "ref.fa", "r1.fq", "r2.fq"], cwd=tmp_path, env=env,
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        assert p.returncode == 0, p.stderr.decode()[-800:]
        out[gpus] = [l for l in p.stdout.split(b"\n") if not l.startswith(b"@PG")]
    assert out["2"] == out["1"] and len(out["1"]) > 60000
