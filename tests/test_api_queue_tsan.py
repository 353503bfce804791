"""mm_map_frag callers of many threads share mini-batches through one request queue per index (airlift_b200/host/apiq.c).
This builds the queue with ThreadSanitizer and a fake batch mapper (tests/aux/apiq_tsan_main.c) and drives it with 32 threads x
2 000 calls of one- and two-segment fragments under three option sets: every caller must get exactly its own hits, no batch may
mix option sets or exceed the base cap, fragments must actually share batches, and stopping the queue must join its thread."""
import os
import re
import shutil
import subprocess
import pytest
import _libs as L


def test_request_queue_under_tsan(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("needs gcc")
    exe = str(tmp_path / "apiq_tsan")
    host = os.path.join(L.ROOT, "airlift_b200", "host")
    cmd = ["gcc", "-O1", "-g", "-fsanitize=thread", "-fno-omit-frame-pointer", "-I" + os.path.join(L.ROOT, "include"), "-I" + host,
           os.path.join(L.ROOT, "tests", "aux", "apiq_tsan_main.c"), os.path.join(host, "apiq.c"), "-o", exe, "-lpthread"]
    b = subprocess.run(cmd, capture_output=True, text=True)
    if b.returncode != 0 and "tsan" in (b.stderr or "").lower():
        pytest.skip("no sanitizer runtime in this toolchain")
    assert b.returncode == 0, b.stderr[-800:]
    r = subprocess.run([exe, "32", "2000"], capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, TSAN_OPTIONS="halt_on_error=0 exitcode=66"))
    assert r.returncode == 0 and "WARNING: ThreadSanitizer" not in r.stderr, r.stderr[-3000:]
    got = {k: int(v) for k, v in re.findall(r"(\w+) (-?\d+)", r.stdout)}
    assert got["calls"] == 64000
    assert got["errors"] == 0, got
    assert got["mixed"] == 0 and got["over_cap"] == 0 and got["bad_opt"] == 0, got
    assert got["multi_frag"] > 0 and got["max_frag"] > 1, got
    assert got["rounds"] < got["calls"], got
    assert got["two_batch_rounds"] > 0, got
    assert got["tasks_running"] == got["tasks_before"] + 1, got
    assert got["tasks_after"] == got["tasks_before"], got
