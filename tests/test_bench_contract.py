"""bench.py's reference arm runs on CPU only: its JSON line must carry the contract's keys (the GPU arm's line is
checked on the GPU box by the driver; here: the parts that need no GPU)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1                                        # ONE JSON line on stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "requests/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["metric"].startswith("agent_requests_per_sec") and d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "requests/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_gojson_string_property():
    """go_string output is always valid JSON whose value is what Go's decoder would give back (hypothesis, CPU)."""
    from hypothesis import given, settings, strategies as st
    sys.path.insert(0, ROOT)
    from oracle import gojson as G

    @settings(max_examples=300, deadline=None)
    @given(st.binary(max_size=64))
    def check(b):
        js = G.go_string(b)
        assert json.loads(js.decode("utf-8")) == G.go_decode(b)
        assert G.go_string(G.go_decode(b)) == G.go_string(G.go_decode(b).encode("utf-8"))   # second marshal is a fixed point
        for ch in (b"<", b">", b"&", b"\xe2\x80\xa8", b"\xe2\x80\xa9"):
            assert ch not in js
    check()


import pytest


def test_bench_arguments_are_checked():
    """--steps sets the number of timed steps (at least one); --dump-outputs covers the GPU path of c2 / c3 only.  Both are
    refused before any work starts, so this runs without a GPU."""
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"], ["--workload", "c5", "--dump-outputs", "out"]):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert res.returncode == 2 and "error:" in res.stderr and res.stdout == "", (extra, res.stderr)


@pytest.mark.gpu
def test_dump_outputs_are_the_same_in_every_run(tmp_path):
    """--dump-outputs writes the verdicts of the last timed step, and two runs with the same arguments write the same
    arrays (seeded records, fixed key of the minted ids)."""
    import numpy as np
    sys.path.insert(0, ROOT)
    from agentainer_lab_b200 import constants as K
    runs = []
    for k in range(2):
        out = tmp_path / f"run{k}"
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-other-mode", "--no-callers",
                              "--no-secondary", "--no-cpu", "--e2e-steps", "1", "--dump-outputs", str(out)],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert res.returncode == 0, res.stderr[-2000:]
        assert json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][0])["steps"] == 2
        runs.append({p.name: np.load(p) for p in out.iterdir()})
    a, b = runs
    assert sorted(a) == ["verdict_agent_slot.npy", "verdict_code.npy", "verdict_flags.npy", "verdict_http_status.npy"]
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for name, x in a.items():
        assert x.dtype == np.float64 and x.shape == (1 << 20,) and np.array_equal(x, b[name]), name
    # C3: every agent is running, so every request is forwarded; ~10 % are replay-flagged, every other one is stored and tracked
    assert (a["verdict_code.npy"] == K.AGR_V_FORWARD).all() and (a["verdict_http_status.npy"] == 0).all()
    flags = a["verdict_flags.npy"].astype(np.int64)
    replay = (flags & K.AGR_VF_REPLAY) != 0
    assert 0.05 < replay.mean() < 0.15
    assert ((flags[~replay] & (K.AGR_VF_STORED | K.AGR_VF_TRACKED)) == (K.AGR_VF_STORED | K.AGR_VF_TRACKED)).all()
    assert len(np.unique(a["verdict_agent_slot.npy"])) <= 256


@pytest.mark.gpu
def test_gpu_arm_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "4", "--warmup", "3", "--no-other-mode", "--no-callers", "--e2e-steps", "2"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "roofline", "e2e", "gpu_launches", "clocks", "cpu_baseline"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 4 and d["warmup"] == 3 and d["scaling"] == "weak" and d["vs_baseline"] is None
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0.3 < r["frac"] < 1.2
    assert "NOT measured in this run" in r["traffic_source"] or r["traffic"] is None
    assert "Zipf" in d["config"]["workload"]                        # the headline is the configuration with duplicate idempotency keys
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 512 * d["config"]["records_per_step_per_gpu"] and e["d2h_bytes_per_step"] > 0
    assert 0 < e["value"] < d["value"]                             # the host link binds end to end
    assert d["gpu_launches"] >= 2 * d["steps"]
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert "sm_mhz" in d["clocks"] and isinstance(d["clocks"]["reasons"], list)
    for k in ("k2_complete", "k3_replay_scan", "k5_json", "sustained_ring"):
        assert k in d["secondary_kernels"]


def test_nccl_banner_is_kept_off_stdout(tmp_path):
    """N > 1: NCCL prints its version banner to file descriptor 1 when torch.distributed creates the communicator; bench.py
    points fd 1 at stderr for that moment and restores it (ONE JSON line on stdout).  Checked with a stand-in for
    torch.distributed in a child process whose stdout is a file."""
    code = r'''
import os, sys
sys.path.insert(0, %r)
import bench
class Dist:
    def init_process_group(self, backend, device_id=None):
        os.write(1, b"NCCL version 0.0.0+test\n")          # what libnccl does: a raw write to fd 1
    def barrier(self): pass
class Cuda:
    def synchronize(self): pass
class Torch:
    cuda = Cuda()
    def device(self, *a): return None
print("before")
bench.init_nccl_quietly(Dist(), Torch(), 0)
print("after")
''' % ROOT
    out, err = tmp_path / "out.txt", tmp_path / "err.txt"
    with open(out, "w") as fo, open(err, "w") as fe:
        res = subprocess.run([sys.executable, "-c", code], stdout=fo, stderr=fe, timeout=120, cwd=ROOT)
    assert res.returncode == 0, err.read_text()
    assert out.read_text().split() == ["before", "after"]
    assert "NCCL version" in err.read_text()


def test_clock_sampler_source_is_valid_and_self_terminating():
    import ast
    sys.path.insert(0, ROOT)
    import bench
    ast.parse(bench.SAMPLER_SRC)
    assert "getppid" in bench.SAMPLER_SRC                           # a killed bench must not leave an NVML poller behind
