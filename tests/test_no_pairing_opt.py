"""CPU-only: mm_b200_check_opt accepts --no-pairing (MM_F_INDEPEND_SEG) and still refuses, with the same message, every mode
this build does not implement."""
import ctypes as C
import os
import subprocess
import pytest
import _libs as L

LIB = os.path.join(L.ROOT, "airlift_b200", "libmm2b200.so")
MM_F_NO_DIAG, MM_F_NO_DUAL, MM_F_SPLICE, MM_F_INDEPEND_SEG = 0x001, 0x002, 0x080, 0x20000


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(LIB):
        subprocess.check_call(["make", "-C", L.ROOT, "lib"])
    import bench
    lib = C.CDLL(LIB)
    lib.mm_set_opt.argtypes = [C.c_char_p, C.POINTER(bench.IdxOpt), C.POINTER(bench.MapOptFull)]
    lib.mm_b200_check_opt.argtypes = [C.POINTER(bench.MapOptFull)]
    return lib


def _opt(lib, preset=b"sr"):
    import bench
    ipt, opt = bench.IdxOpt(), bench.MapOptFull()
    lib.mm_set_opt(None, C.byref(ipt), C.byref(opt))
    lib.mm_set_opt(preset, C.byref(ipt), C.byref(opt))
    return opt


@pytest.mark.parametrize("preset", [b"sr", b"map-ont"])
def test_no_pairing_is_accepted(lib, preset):
    opt = _opt(lib, preset)
    assert lib.mm_b200_check_opt(C.byref(opt)) == 0
    opt.flag |= MM_F_INDEPEND_SEG
    assert lib.mm_b200_check_opt(C.byref(opt)) == 0


def _refused(lib, change):
    opt = _opt(lib)
    opt.flag |= MM_F_INDEPEND_SEG
    change(opt)
    return lib.mm_b200_check_opt(C.byref(opt))


@pytest.mark.parametrize("what,change", [
    ("splice", lambda o: setattr(o, "flag", o.flag | MM_F_SPLICE)),
    ("-D", lambda o: setattr(o, "flag", o.flag | MM_F_NO_DIAG)),
    ("-X", lambda o: setattr(o, "flag", o.flag | MM_F_NO_DIAG | MM_F_NO_DUAL)),
    ("--dual=no", lambda o: setattr(o, "flag", o.flag | MM_F_NO_DUAL)),
    ("-T", lambda o: setattr(o, "sdust_thres", 20)),
    ("--split-prefix", lambda o: setattr(o, "split_prefix", b"prefix")),
], ids=lambda x: x if isinstance(x, str) else "")
def test_other_modes_still_refused(lib, what, change):
    assert _refused(lib, change) == -1


def test_refusal_messages(tmp_path):
    """the CLI takes --no-pairing past the option check; the remaining refusals keep their wording"""
    cli = os.path.join(L.ROOT, "build", "minimap2-b200")
    if not os.path.exists(cli):
        pytest.skip("needs build/minimap2-b200")
    fa = tmp_path / "missing.fa"
    p = subprocess.run([cli, "-ax", "sr", "--no-pairing", str(fa), str(fa)], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert b"not supported by this build" not in p.stderr
    assert b"failed to open file" in p.stderr  # it got as far as opening the index
    cases = {("-ax", "splice"): b"[ERROR] spliced alignment (--splice, ksw_exts2) is not supported by this build",
             ("-ax", "sr", "-T", "20"): b"[ERROR] SDUST masking of query minimizers (-T, map.c:41-62) is not supported by this build",
             ("-ax", "sr", "--dual=no"): b"[ERROR] the self/dual-hit filters of the all-vs-all modes (-D, -X, --dual=no, ava-ont, ava-pb; map.c:128-137) is not supported by this build"}
    for args, msg in cases.items():
        p = subprocess.run([cli] + list(args) + [str(fa), str(fa)], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        assert p.returncode != 0 and msg in p.stderr, (args, p.stderr[-400:])
