"""Runs of ring slots (variable-length records through the single-request front end): the run-aware callers' side of
csrc/agr_ring.hpp against a stand-in for the dispatcher and the service kernel, on the CPU (tests/ring_sim_var.cpp).  Records of
96 B .. 8192 B take 1 .. 16 consecutive slots next to one-slot operations; every operation must be answered exactly once from
all the slots of its own run, runs must be consumed whole, oversubscribed ticket holders must finish, and runs cross the ring's
end."""
import json
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "ring_sim_var.cpp")


@pytest.fixture(scope="module")
def ring_sim_var(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("ringvar") / "ring_sim_var")
    res = subprocess.run(["g++", "-O2", "-std=c++17", "-pthread", "-Wall", "-o", exe, SRC], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr
    return exe


def _run(exe, args, timeout):
    res = subprocess.run([exe, *args], capture_output=True, text=True, timeout=timeout)      # a deadlock shows up as the timeout
    d = json.loads(res.stdout.strip().splitlines()[-1])
    assert res.returncode == 0 and d["ok"] and d["wrong_answers"] == 0 and d["torn_runs"] == 0 and d["served"] == d["operations"], d
    return d


@pytest.mark.parametrize("args", [
    ("2", "0", "0", "20000"),                 # blocking callers only: records and outcomes alternate
    ("0", "4", "512", "40000"),               # ticket callers, well inside the ring
    ("0", "8", "2048", "20000", "20"),        # 8 x 2048 parked tickets of up to 16 slots each against 16384 slots
    ("2", "6", "1024", "20000", "3"),         # blocking and ticket callers on one ring, oversubscribed
])
def test_ring_runs_on_cpu(ring_sim_var, args):
    d = _run(ring_sim_var, args, 300)
    assert d["longest_run"] == 16 and d["runs_across_ring_end"] > 0 and d["ring_laps"] > 3, d
    if int(args[1]) * int(args[2]) > 16384 // 8:
        assert d["eagain"] > 0 and d["skipped_slots"] > 0, d           # the oversubscribed runs really went through the no-op path


def test_ring_runs_under_thread_sanitizer(tmp_path):
    """The same simulation built with -fsanitize=thread: the run-aware caller code (streaming stores behind an sfence, the length
    word, continuation ready words before the head's release store) has no data race ThreadSanitizer can see."""
    exe = str(tmp_path / "ring_sim_var_tsan")
    res = subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-pthread", "-fsanitize=thread", "-o", exe, SRC], capture_output=True, text=True, timeout=300)
    if res.returncode != 0:
        pytest.skip("no ThreadSanitizer runtime in this image: " + res.stderr[-200:])
    assert "-Wtsan" not in res.stderr
    for args in (("1", "3", "256", "4000"), ("1", "6", "2048", "3000", "20")):
        run = subprocess.run([exe, *args], capture_output=True, text=True, timeout=600)
        assert "ThreadSanitizer" not in run.stderr, run.stderr[-2000:]
        d = json.loads(run.stdout.strip().splitlines()[-1])
        assert run.returncode == 0 and d["ok"], d
