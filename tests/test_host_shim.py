"""The C++17 host-side mirror of the reference handlers (gyeeta_b200/host/gy_gysk_shim.h) compiles with g++ against the C ABI
and links libgysketch.so. CPU: creating an engine fails loudly, handlers return false. GPU: the same binary ingests a
TCP_CONN_NOTIFY / AGGR_TASK_STATE_NOTIFY batch and reads the summary back."""
import os
import subprocess

import pytest

from gyeeta_b200 import engine as ge

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(outdir):
    """the test binaries go to a temporary directory: the repository tree may be read-only"""
    src = os.path.join(ROOT, "tests", "cpp", "shim_smoke.cc")
    exe = os.path.join(str(outdir), "shim_smoke")
    libdir = os.path.dirname(ge.LIB_PATH)
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "gyeeta_b200", "host"),
           "-I", os.path.join(ROOT, "gyeeta_b200", "csrc"), src, "-o", exe, "-L", libdir, "-lgysketch", f"-Wl,-rpath,{libdir}"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_shim_compiles_and_fails_loudly_without_gpu(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu test")
    r = subprocess.run([_build(tmp_path)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "rc=-19" in r.stdout and "handlers: 0 0 0" in r.stdout and "more handlers: 0 0 0" in r.stdout and "tick: 0 deletes: 0 records: -1" in r.stdout


@pytest.mark.gpu
def test_shim_end_to_end_on_gpu(tmp_path):
    r = subprocess.run([_build(tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "handlers: 1 1 1" in r.stdout and "more handlers: 1 1 1" in r.stdout and "found=1 nconns_5s=1 kbytes_5s=4" in r.stdout
    assert "nconns_active=3 active_kbytes=10 max_rtt=1.5" in r.stdout and "stats: resp=1 tcp=3 svcs=3" in r.stdout


def test_wire_validators_accept_and_reject_like_the_reference(tmp_path):
    """gysk_wire.h's validate_batch against hand-built batches, the rules of TCP_CONN_NOTIFY::validate /
    AGGR_TASK_STATE_NOTIFY::validate / LISTENER_STATE_NOTIFY::validate (common/gy_comm_proto.cc:840-996): element sizes multiples
    of 8 and inside the message, at most MAX elements, success iff all were walked, strings NUL-forced in place. Pure host code."""
    src = os.path.join(ROOT, "tests", "cpp", "wire_validate.cc")
    exe = os.path.join(str(tmp_path), "wire_validate")
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "gyeeta_b200", "csrc"), src, "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and "failures: 0" in r.stdout and "MISMATCH" not in r.stdout, r.stdout
