"""Every reference citation (file.go:line[-line]) in the header, the oracle and the design documents must point into a file
that exists in the reference tree and at lines that exist in it.  The reference's line counts are stored in
tests/golden/reference_line_counts.json (taken from the cited commit), so the check needs no copy of the reference."""
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LINE_COUNTS = os.path.join(ROOT, "tests", "golden", "reference_line_counts.json")
FILES = ["include/agentainer_gpu.h", "DESIGN.md", "INTEGRATION.md", "oracle/model.py", "oracle/gojson.py", "oracle/cpu_ref.c",
         "agentainer-lab_b200/host/requests.hpp", "agentainer-lab_b200/host/requests.cpp", "agentainer-lab_b200/csrc/agr_k5_json.cu",
         "agentainer-lab_b200/csrc/agr_kernels.cu", "agentainer-lab_b200/csrc/agr_device.cuh", "agentainer-lab_b200/csrc/agr_json_host.cpp"]
KNOWN = {"requests.go": "internal/requests/requests.go", "replay_worker.go": "internal/requests/replay_worker.go",
         "server.go": "internal/api/server.go", "agent.go": "internal/agent/agent.go", "main.go": "cmd/agentainer/main.go",
         "storage.go": "internal/storage/storage.go", "state_sync.go": "internal/sync/state_sync.go",
         "quick_sync.go": "pkg/agentsync/quick_sync.go", "config.go": "internal/config/config.go"}


def test_citations_point_at_existing_lines():
    with open(LINE_COUNTS) as f:
        counts = json.load(f)["lines"]
    lengths = {short: counts[rel] for short, rel in KNOWN.items() if rel in counts}
    assert {"requests.go", "replay_worker.go", "server.go", "agent.go"} <= set(lengths)
    bad, seen = [], 0
    pat = re.compile(r"\b(?:[A-Za-z_./-]*/)?([a-z_]+\.go):(\d+)((?:[-,]\d+)*)")
    for rel in FILES:
        text = open(os.path.join(ROOT, rel), errors="replace").read()
        for m in pat.finditer(text):
            name = m.group(1)
            if name not in lengths:
                continue
            nums = [int(m.group(2))] + [int(x) for x in re.findall(r"\d+", m.group(3))]
            seen += 1
            if max(nums) > lengths[name] or min(nums) < 1:
                bad.append((rel, m.group(0), lengths[name]))
    assert seen > 150
    assert not bad, bad[:10]
