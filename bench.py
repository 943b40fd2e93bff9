#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (BASELINE.json): agent requests/sec through
ingest + dedupe + route on 512 B records.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c2|c5] [--dump-outputs DIR]

A "step" is ONE pass of the hot path (K1: ingest + dedupe + route) over ONE batch of the workload's records.  The
headline workload is c3 = BASELINE configs[2], the largest single-GPU configuration and the one with duplicate
idempotency keys (10 M+ records in 1 M-record steps, 256 agent ids Zipf s = 1.2, 10 % replay-flagged duplicates);
c2 = configs[1] (1 M records, uniform, no duplicates) and both id modes are reported next to it under "configs".
  value     whole-job records/s, records already resident in the HBM slab when the timed region starts
            (CUDA events on the engine's stream, barrier + synchronize on both sides, max over ranks);
  e2e       the same metric through the C-ABI call a host makes (agr_ingest) with PINNED HOST buffers: the
            host->device copy of the step's records and the device->host read of its verdicts are inside the
            timed region;
  roofline  dominant kernel (k1_ingest): algorithmic bytes (520 B/record, SURVEY 8d) / its device time measured
            live with CUDA events on the launching stream, against MEASURED_PEAKS.json hbm_gbs;
  cpu_baseline  the C restatement of the reference's Go+Redis path (oracle/cpu_ref.c, kind "port": the reference
            itself cannot be built in this image) timed on ONE host core over a bounded sample.
  --impl reference  times that CPU restatement on all host threads (agents sharded across threads) on the same
            workload/metric — the reference arm the driver compares against.
  --dump-outputs DIR  after the timed steps, the verdicts of the last one as DIR/verdict_<field>.npy (float64).  The
            records are seeded and the key of the minted ids is fixed, so the same arguments give the same inputs in every
            run and two builds can be compared output for output.
Under torchrun (N > 1) every rank owns one GPU and one shard of the agents; no data-path collective is needed
for c2/c3 (records are steered to the owner shard before the copy), so scaling is "weak".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the bench runs from a built tree that may be read-only: it leaves no __pycache__ there

METRIC = "agent_requests_per_sec_ingest_dedupe_route_512B"
ALG_BYTES_PER_RECORD = 520          # SURVEY.md 8(d): 512 B record read + 4 B queue/state entry + 4 B verdict
ID_SECRET = 0x9E3779B97F4A7C15      # key of the engine-minted ids of the headline run (AGR_CFG_MINT_IDS)
WORKLOADS = {
    "c2": dict(name="C2: 1M synthetic 512B POST /agent/<id>/chat records per step, 256 agent ids, uniform, all agents running, no crash-replay",
               records=1 << 20, agents=256, zipf_milli=0, dup_permille=0),
    "c3": dict(name="C3: 1M-record steps of the 10M+ record stream, 256 agent ids Zipf s=1.2, 10% replay-flagged duplicates (duplicate idempotency keys: replay_of names an earlier request of the same agent)",
               records=1 << 20, agents=256, zipf_milli=1200, dup_permille=100),
}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def k1_traffic(mode, variant):
    """DRAM bytes per K1 launch from the committed ncu capture of the same kernel and batch size.  NOT measured in this run:
    ncu replays the kernel ~40 times and a number printed under it is no bench value; the source file is named."""
    tp = os.path.join(ROOT, "profiles", "k1_traffic.json")
    try:
        doc = json.load(open(tp))
        e = doc.get(f"{mode}_variant{variant}", {})
        return e.get("dram_bytes_per_launch"), f"profiles/k1_traffic.json <- {e.get('source', doc.get('_source', 'ncu --set full capture'))} (read from the committed file, NOT measured in this run)"
    except Exception:
        return None, "no committed ncu capture for this mode"


def init_nccl_quietly(dist, torch, local_rank):
    """NCCL prints its version banner to STDOUT when the first communicator comes up; the contract is ONE JSON line there, so
    file descriptor 1 points at stderr while torch.distributed creates its communicator (eagerly: device_id is given)."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
        torch.cuda.synchronize()
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)



def run_callers(local_rank, seconds=2.0):
    """e2e_callers: the reference's real call pattern (one request per call, server.go:493) through the C-ABI, measured by the
    C++ driver host/bench_callers in its own process: blocking agr_ingest_ex(n=1) + agr_complete(n=1) from T OS threads, and
    the ticket form (agr_submit_* / agr_poll) with many requests parked per thread."""
    import agentainer_lab_b200 as A
    exe = os.path.join(os.path.dirname(A.build_host()), "bench_callers")
    out = {"unit": "round trips/s (one StoreRequest+decision and one StoreResponse each)", "blocking": {}, "tickets": {}}
    try:
        quota = open("/sys/fs/cgroup/cpu.max").read().split()
        out["host_cpu_allowance"] = (os.cpu_count() if quota[0] == "max" else int(quota[0]) / int(quota[1]))
    except Exception:
        out["host_cpu_allowance"] = os.cpu_count()
    def one(threads, inflight):
        try:
            r = subprocess.run([exe, str(threads), str(seconds), str(local_rank), "mint", "256", str(inflight)], capture_output=True, text=True, timeout=90)
            return json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:
            return {"error": repr(e)}
    for t in (8, 64, 256):
        out["blocking"][f"threads_{t}"] = one(t, 0)
    for t, w in ((4, 512), (8, 512), (12, 256)):
        out["tickets"][f"threads_{t}_inflight_{w}"] = one(t, w)
    best = max((v.get("round_trips_per_s", 0), k, v) for d in (out["blocking"], out["tickets"]) for k, v in d.items())
    out["value"], out["best"] = best[0], best[1]
    out["p50_us"], out["p99_us"] = best[2].get("p50_us"), best[2].get("p99_us")
    return out


SAMPLER_SRC = """
import sys, time
import pynvml as N
N.nvmlInit()
h = N.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))
get_reasons = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
out = open(sys.argv[2], "w", buffering=1)
print("max", N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM), file=out)
import os
parent, t_end, k = int(sys.argv[3]), time.time() + 600.0, 0
while True:
    print("%.6f" % time.time(), N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM), get_reasons(h), file=out)
    time.sleep(0.0002)
    k += 1
    if k % 512 == 0 and (os.getppid() != parent or time.time() > t_end):    # never outlive the bench (a killed parent cannot stop us)
        break
"""


class ClockSampler:
    """SM clock / clock-event reasons sampled through NVML by a SEPARATE process (NVML calls made from a process with a
    busy CUDA context stall for milliseconds), ~5 kHz, wall-clock timestamps; the timed region is a few ms long."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int):
        import tempfile
        self.index, self.proc, self.t0, self.t1 = index, None, 0.0, float("inf")
        self.path = os.path.join(tempfile.gettempdir(), f"agr_clocks_{os.getpid()}_{index}.txt")

    def start(self):
        try:
            self.proc = subprocess.Popen([sys.executable, "-c", SAMPLER_SRC, str(self.index), self.path, str(os.getpid())],
                                         stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def wait_ready(self, timeout=10.0):
        """block until the sampler process has written its first sample (it needs ~0.5 s to import NVML)"""
        t = time.time()
        while time.time() - t < timeout:
            try:
                if os.path.getsize(self.path) > 64:
                    return True
            except OSError:
                pass
            time.sleep(0.01)
        return False

    def mark(self):
        self.t0 = time.time()

    def unmark(self):
        self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "error": "sampler did not start"}
        time.sleep(0.01)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        mx, rows = None, []
        try:
            for ln in open(self.path):
                f = ln.split()
                if f and f[0] == "max":
                    mx = float(f[1])
                elif len(f) == 3:
                    rows.append((float(f[0]), float(f[1]), int(f[2])))
            os.remove(self.path)
        except Exception as e:
            return {"sm_mhz": None, "sm_max_mhz": mx, "reasons": [], "samples": 0, "error": repr(e)}
        timed, scope = [r for r in rows if self.t0 <= r[0] <= self.t1], "timed region"
        if len(timed) < 3:
            timed, scope = [r for r in rows if self.t0 - 0.02 <= r[0] <= self.t1 + 0.02], "timed region +/- 20 ms"
        if not timed:
            return {"sm_mhz": None, "sm_max_mhz": mx, "reasons": [], "samples": 0, "error": "no NVML sample near the timed region"}
        reasons = 0
        for r in timed:
            reasons |= r[2]
        return {"sm_mhz": float(np.median([r[1] for r in timed])), "sm_max_mhz": mx,
                "reasons": sorted(v for k, v in self.REASONS.items() if reasons & k), "samples": len(timed), "scope": scope}


def parallel_fill(A, out, first_index, wl, seed, nanos0, threads=16, mint=None):
    n = len(out)
    per = (n + threads - 1) // threads
    ts = []
    for t in range(threads):
        a, b = t * per, min(n, (t + 1) * per)
        if a >= b:
            break
        th = threading.Thread(target=A.synth_fill_host, args=(first_index + a, b - a),
                              kwargs=dict(seed=seed, n_agents=wl["agents"], zipf_milli=wl["zipf_milli"],
                                          dup_permille=wl["dup_permille"], agent_nanos0=nanos0, mint=mint, out=out[a:b]))
        th.start(); ts.append(th)
    for th in ts:
        th.join()


# --------------------------------------------------------------------------------------------- CPU arms
def cpu_port_single(A, wl, budget_s=12.0, max_records=3_000_000):
    """oracle/cpu_ref.c (restatement of the Go+Redis path) on ONE core over a bounded sample of the workload."""
    from oracle.cpu_ref import CRef
    chunk = 1 << 16
    c = CRef()
    for k in range(wl["agents"]):
        c.set_agent_state(A.synth_agent_id(k), "running")
    done, spent = 0, 0.0
    while spent < budget_s and done < max_records:
        recs = A.synth_fill_host(done, chunk, seed=2, n_agents=wl["agents"], zipf_milli=wl["zipf_milli"], dup_permille=wl["dup_permille"])
        t = time.perf_counter()
        c.ingest(recs)
        spent += time.perf_counter() - t
        done += chunk
    c.close()
    return {"value": done / spent, "unit": "requests/s", "cores": 1, "kind": "port",
            "sample": f"first {done} records of the workload stream, ingest+dedupe+route only (GetAgent + StoreRequest + status gate with JSON/base64 marshal, no RESP/TCP), {spent:.1f} s"}


def _ref_worker(p, T, wl, per_step, steps, warmup, barrier, q):
    """One shard of the CPU restatement: owns agents p, p+T, ... (agents are independent in the reference: every key
    is agent:{id}:...), gets its share of every step's records, and times only the ingest+dedupe+route calls."""
    import agentainer_lab_b200 as A
    from oracle.cpu_ref import CRef
    na = wl["agents"] // T
    nanos0 = 1700000000000000000 + p * 1_000_000_000
    c = CRef()
    for k in range(na):
        c.set_agent_state(A.synth_agent_id(k, agent_nanos0=nanos0), "running")
    m = per_step // T
    times = []
    for step in range(warmup + steps):
        recs = A.synth_fill_host(step * m, m, seed=100 + p, n_agents=na, zipf_milli=wl["zipf_milli"],
                                 dup_permille=wl["dup_permille"], agent_nanos0=nanos0)
        barrier.wait()
        t0 = time.perf_counter()
        v, _ = c.ingest(recs)
        dt = time.perf_counter() - t0
        barrier.wait()
        if step >= warmup:
            times.append(dt)
    assert (v["code"] == 1).all()
    q.put(times)


def run_reference(args, wl, rank, world):
    """--impl reference: the CPU restatement of the Go+Redis path on all the host cores it can use.  The reference
    itself serialises on ONE Redis thread; here agents are sharded over T independent processes (each with its own
    mini-Redis), which can only flatter it.  Each step is the full workload batch split over the shards."""
    import multiprocessing as mp
    if rank != 0:
        return
    ncpu = os.cpu_count() or 1
    T = max(t for t in (1, 2, 4, 8, 16, 32, 64) if t <= ncpu and wl["agents"] % t == 0)
    per_step = wl["records"] if T >= 16 else wl["records"] // 8
    ctx = mp.get_context("fork")
    barrier, q = ctx.Barrier(T), ctx.Queue()
    procs = [ctx.Process(target=_ref_worker, args=(p, T, wl, per_step, args.steps, args.warmup, barrier, q)) for p in range(T)]
    for pr in procs:
        pr.start()
    all_times = [q.get() for _ in procs]
    for pr in procs:
        pr.join()
    step_times = [max(t[i] for t in all_times) for i in range(args.steps)]      # a step ends when its slowest shard ends
    total = sum(step_times)
    val = per_step * args.steps / total
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "requests/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": wl["name"], "records_per_step": per_step, "agents": wl["agents"]},
            "cpu_baseline": {"value": val, "unit": "requests/s", "cores": T, "kind": "port",
                             "sample": f"{per_step} records per step, agents sharded over {T} processes of oracle/cpu_ref.c (reference Go+Redis cannot be built here: no go, no redis-server)"},
            "e2e": {"value": val, "unit": "requests/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------- GPU arm
def measure_resident(A, K, torch, dist, args, wl, rank, local_rank, extra_flags, steps, warmup):
    """Device-resident K1 measurement on a fresh engine: records pre-generated in the slab, `steps` timed launches."""
    B = wl["records"]
    eng = A.Engine(device=local_rank, slab_rows=(warmup + steps) * B, max_agents=1024, max_batch=B, k1_variant=args.variant | (args.timing_stride << 16),
                   flags=K.AGR_CFG_PERSISTENCE | K.AGR_CFG_TIMING | extra_flags)
    nanos0 = 1700000000000000000 + rank * 10_000_000_000
    for k in range(wl["agents"]):
        eng.set_agent_state(A.synth_agent_id(k, agent_nanos0=nanos0), "running")
    synth = dict(seed=2 + rank, n_agents=wl["agents"], zipf_milli=wl["zipf_milli"], dup_permille=wl["dup_permille"], agent_nanos0=nanos0)
    first = eng.reserve_rows(B)
    for s in range(1, warmup + steps):
        eng.reserve_rows(B)
    mint_base = first if (extra_flags & K.AGR_CFG_MINT_IDS) else None
    for s in range(warmup + steps):
        eng.synth_fill_rows(s * B, first + s * B, B, mint_base=mint_base, **synth)
    stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", local_rank))
    for s in range(warmup):
        eng.ingest_rows_async(first + s * B, B)
    eng.sync(); eng.kernel_time()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    ev0.record(stream)
    for s in range(warmup, warmup + steps):
        eng.ingest_rows_async(first + s * B, B)
    ev1.record(stream)
    eng.sync(); torch.cuda.synchronize()
    dev_ms = ev0.elapsed_time(ev1)
    k_ms, k_n = eng.kernel_time()
    st = eng.stats()
    assert st["stored"] + st["replay_flagged"] == (warmup + steps) * B, st
    eng.close()
    return dev_ms, k_ms / max(1, k_n)


def measure_sustained(A, K, torch, local_rank, variant, steps=48):
    """The ring under load (AGR_CFG_RING): 1 M records per step through an 8 M-row slab, every record left pending and
    dropped by the key TTL four steps later; each step = K1 over the batch + agr_expire + agr_reclaim.  Device time per step
    from CUDA events around those three calls (the record generator that refills the rows is outside them)."""
    B = 1 << 20
    R = 8 * B
    eng = A.Engine(device=local_rank, slab_rows=R, max_agents=1024, max_batch=B, k1_variant=variant,
                   flags=K.AGR_CFG_PERSISTENCE | K.AGR_CFG_MINT_IDS | K.AGR_CFG_RING)
    nanos0 = 1700000000000000000
    names = [A.synth_agent_id(k, agent_nanos0=nanos0) for k in range(256)]
    eng.set_agent_states(names, ["stopped"] * 256)
    synth = dict(seed=11, n_agents=256, agent_nanos0=nanos0)
    stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", local_rank))
    warm = 10
    evs = [tuple(torch.cuda.Event(enable_timing=True) for _ in range(4)) for _ in range(steps)]
    released = 0
    for s in range(warm + steps):
        first = eng.reserve_rows(B)
        eng.synth_fill_rows(s * B, first, B, **synth)           # seq of record j = its stream index: the clock of this run
        if s >= warm:
            evs[s - warm][0].record(stream)
        eng.ingest_rows_async(first, B)
        if s >= warm:
            evs[s - warm][1].record(stream)
        eng.expire((s + 1) * B, 4 * B, want_count=False)           # enqueue the TTL sweep ...
        if s >= warm:
            evs[s - warm][2].record(stream)
        released += eng.reclaim_async()                             # ... release what the previous step's scan found, start the next scan
        if s >= warm:
            evs[s - warm][3].record(stream)
    eng.sync(); torch.cuda.synchronize()
    ms = sum(e[0].elapsed_time(e[3]) for e in evs) / steps
    parts = [sum(e[k].elapsed_time(e[k + 1]) for e in evs) / steps for k in range(3)]
    st = eng.stats()
    assert st["stored"] == (warm + steps) * B and st["rows_used"] == (warm + steps) * B, st
    assert st["rows_used"] - st["rows_tail"] <= R and released >= (warm + steps - 6) * B, (st, released)
    eng.close()
    return {"records_per_step": B, "ring_rows": R, "steps": steps, "laps": (warm + steps) * B / R, "ms_per_step": ms,
            "requests_per_s": B / (ms * 1e-3), "rows_released": released,
            "ms_by_call": {"ingest (K1 + k1_post)": parts[0], "agr_expire": parts[1], "agr_reclaim_async": parts[2]},
            "what": "K1 + agr_expire (TTL sweep: per-chunk time bounds, only due chunks are read) + agr_reclaim_async (release of 1 M rows, one step behind, no host wait) per step, device time"}


def bind_to_gpu_numa_node(index: int):
    """Run on (and therefore allocate pinned host memory from) the CPUs NVML reports as local to the GPU: DMA from the far
    socket of a two-socket host loses ~25 % of the PCIe bandwidth.  A host process serving one GPU would be pinned the same way."""
    if os.environ.get("AGR_NO_AFFINITY"):
        return None
    try:
        import pynvml as N
        N.nvmlInit()
        h = N.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = N.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        cpus &= set(range(ncpu))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def verify_exchange(A, K, dist, rank, world, local_rank):
    """Driver-visible correctness of the multi-GPU path: tests/sharded_check.py (the body of tests/test_sharded_gpu.py, which
    the driver's one-GPU test box skips) on a fresh engine per rank — every record's verdict wherever it was decided and every
    owner's per-agent pending / completed / failed lists against oracle/cpu_ref.c fed the owner's merge order.  The oracle is the
    CHECKER here, outside every timed region.  A mismatch fails the run."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from sharded_check import check_sharded
    import torch
    r = check_sharded(A, K, dist, rank, world, device=local_rank)
    t = torch.tensor([1.0 if r["ok"] else 0.0, r["verdicts_checked"], r["agent_lists_checked"]], device="cuda", dtype=torch.float64)
    dist.all_reduce(t)
    res = {"ok": bool(t[0].item() == world), "ranks": world, "verdicts_checked": int(t[1].item()), "agent_lists_checked": int(t[2].item()),
           "oracle": "oracle/cpu_ref.c (CRef), owner merge order = own host first, then peers by rank"}
    if not res["ok"]:
        print(json.dumps({"error": "sharded results differ from the oracle", **res}), file=sys.stderr)
        sys.exit(3)
    return res


def run_c4(args, rank, world, local_rank):
    """--workload c4 (BASELINE configs[3]): 10 M records per GPU in 1 M-record steps, sharded by FNV-1a64(agent_id) mod N; 95 % of
    a rank's batch are fresh records of its own agents, 5 % are replay-flagged records whose agent lives on another shard ->
    K4 + NCCL all-to-all + K1 at the owner.  value = the exchange with the batch resident in HBM (agr_ingest_sharded_rows),
    e2e = agr_ingest_sharded from pinned host buffers."""
    import torch
    import torch.distributed as dist
    import agentainer_lab_b200 as A
    from agentainer_lab_b200 import constants as K
    from agentainer_lab_b200.sharding import owned_agents, make_rank_batch
    torch.cuda.set_device(local_rank)
    if world > 1:
        init_nccl_quietly(dist, torch, local_rank)
    else:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1"); os.environ.setdefault("MASTER_PORT", "29533")
        dist.init_process_group("gloo", rank=0, world_size=1)
    local_cpus = bind_to_gpu_numa_node(local_rank)
    B, W = 1 << 20, args.warmup
    S = args.steps if args.steps is not None else 10             # 10 x 1 M = 10 M records per GPU unless --steps says otherwise
    e_steps, e_warm = min(S, args.e2e_steps), 1
    rows = int((W + S + e_warm + e_steps + 1) * B * 1.1)
    eng = A.Engine(device=local_rank, slab_rows=rows, max_agents=1024, max_batch=B, k1_variant=args.variant,
                   flags=K.AGR_CFG_PERSISTENCE | K.AGR_CFG_TIMING | K.AGR_CFG_MINT_IDS)
    sys.stdout.flush()
    saved_stdout = os.dup(1); os.dup2(2, 1)                      # NCCL prints its banner to stdout
    try:
        uid = [A.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        eng.comm_init(uid[0], rank, world)
    finally:
        os.dup2(saved_stdout, 1); os.close(saved_stdout)
    own = owned_agents(world, 64, nanos0=1800000000000000000)
    for a in own[rank]:
        eng.set_agent_state(a, "running")
    pins = [eng.pinned(B), eng.pinned(B)]
    firsts = []
    for s in range(W + S):                                       # the batches are resident in their slab rows before the timed region
        pins[0].array[:] = make_rank_batch(rank, world, own, B, seed=70 + s, p_cross_replay=0.05, first_index=s * B)
        f = eng.reserve_rows(B); eng.fill_rows(f, pins[0].array); firsts.append(f)
    stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", local_rank))
    for s in range(W):
        eng.ingest_sharded_rows(firsts[s], B)
    eng.kernel_time()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.barrier(); torch.cuda.synchronize()
    sent = recvd = 0
    t0 = time.perf_counter()
    ev0.record(stream)
    for s in range(W, W + S):
        _, info = eng.ingest_sharded_rows(firsts[s], B)
        sent += info.n_sent; recvd += info.n_received
    ev1.record(stream)
    eng.sync(); torch.cuda.synchronize()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    dist.barrier()
    dev_ms = ev0.elapsed_time(ev1)
    k_ms, k_n = eng.kernel_time()
    # e2e: host buffers in, verdicts out, two-slot pinned ring
    e_times = []
    pins[0].array[:] = make_rank_batch(rank, world, own, B, seed=200, p_cross_replay=0.05, first_index=(W + S) * B)
    for s in range(e_warm + e_steps):
        if s + 1 < e_warm + e_steps:
            pins[(s + 1) % 2].array[:] = make_rank_batch(rank, world, own, B, seed=201 + s, p_cross_replay=0.05, first_index=(W + S + s + 1) * B)
        dist.barrier()
        t = time.perf_counter()
        xv, info = eng.ingest_sharded(pins[s % 2].array)
        dist.barrier()
        if s >= e_warm:
            e_times.append(time.perf_counter() - t)
    assert (xv["code"] == K.AGR_V_FORWARD).all()
    e_ms = 1e3 * sum(e_times) / len(e_times)
    st = eng.stats()
    eng.close()
    verified = verify_exchange(A, K, dist, rank, world, local_rank) if world > 1 else None
    t_all = torch.tensor([dev_ms, e_ms, k_ms], device="cuda" if world > 1 else "cpu", dtype=torch.float64)
    c_all = torch.tensor([float(sent), float(recvd), float(st["ingested"])], device="cuda" if world > 1 else "cpu", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX); dist.all_reduce(c_all)
    dev_ms, e_ms, k_ms = [float(x) for x in t_all.tolist()]
    if rank == 0:
        peak, peak_src = measured_peak()
        rows_k1 = S * B + float(c_all[1]) / world                 # rows K1 decided on this rank in the timed region (own + received)
        ach = ALG_BYTES_PER_RECORD * rows_k1 / (k_ms * 1e-3) / 1e9
        line = {"metric": METRIC, "value": world * B * S / (dev_ms * 1e-3), "unit": "requests/s", "n_gpus": world, "steps": S, "warmup": W,
                "ms_per_step": dev_ms / S, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
                "config": {"workload": f"C4: {world} x B200 sharded by FNV-1a64(agent_id) mod {world}, {S * B * world} records ({S} steps of 1M per GPU), 5% cross-shard replay-flagged records -> NCCL all-to-all",
                           "records_per_step_per_gpu": B, "agents_per_gpu": 64, "record_bytes": 512, "parallelism": f"shard{world}: K4 bin/pack in place + ONE grouped ncclSend/ncclRecv all-to-all per step + K1 at the owner + verdicts back",
                           "l2": "each step reads a fresh 512 MiB batch (> 126 MB L2); no explicit flush", "id_mode": "mint"},
                "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                             "kernel": "k1_ingest (own rows + received rows)", "kernel_ms": k_ms / max(1, k_n), "launches_timed": k_n,
                             "algorithmic_bytes_per_record": ALG_BYTES_PER_RECORD, "peak_source": peak_src},
                "exchange": {"ms_per_step": dev_ms / S, "cross_shard_fraction": float(c_all[0]) / (world * B * S),
                             "nvlink_bytes_per_step": float(c_all[0]) * (512 + 8) / S, "records_sent_per_step": float(c_all[0]) / S,
                             "verified_against_oracle": verified},
                "e2e": {"value": world * B / (e_ms * 1e-3), "unit": "requests/s", "h2d_bytes_per_step": B * 512, "d2h_bytes_per_step": B * 8,
                        "steps": len(e_times), "ms_per_step": e_ms, "api": "agr_ingest_sharded (pinned host records in, verdicts out)",
                        "host_cpus_local_to_gpu": local_cpus},
                "gpu_launches": S * 9, "wall_ms_timed_region": wall_ms, "device_ms_timed_region": dev_ms}
        print(json.dumps(line))
    dist.destroy_process_group()


def dump_verdicts(out_dir, route):
    """--dump-outputs: the verdicts of one timed step as agr_ingest_rows would hand them to its caller (agr_verdict
    {code, flags, http_status, agent_slot}).  The timed launches leave them on the device as one route word per row
    (slot in bits 0..22, code in 23..25, AGR_VF_* flags from bit 26); the fields are unpacked here the way k1_verdict_word
    does on the device, one float64 array per field (4 x 8 MiB for a 1 M-record step)."""
    from agentainer_lab_b200 import constants as K
    route = route.astype(np.int64)
    code = (route >> 23) & 0x7
    http = np.select([code == K.AGR_V_QUEUED, code == K.AGR_V_UNAVAILABLE, code == K.AGR_V_NOT_FOUND], [202, 503, 404], 0)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("verdict_code", code), ("verdict_flags", route >> 26), ("verdict_http_status", http),
                    ("verdict_agent_slot", route & 0x7FFFFF)):
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def run_ours(args, wl, rank, world, local_rank):
    import torch
    import agentainer_lab_b200 as A
    from agentainer_lab_b200 import constants as K
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        init_nccl_quietly(dist, torch, local_rank)
    local_cpus = bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    sampler = ClockSampler(local_rank)
    sampler.start()
    B, W, S = wl["records"], args.warmup, args.steps
    e_steps, e_warm = min(S, args.e2e_steps), 1
    rows = max(args.rows, (W + S) * B + (e_warm + e_steps) * B + (B if world > 1 else 0) * 2)
    id_flags = K.AGR_CFG_MINT_IDS if args.id_mode == "mint" else 0
    # a fixed id key: the minted ids, and with them the records that name them and the verdicts, are the same in every run
    eng = A.Engine(device=local_rank, slab_rows=rows, max_agents=1024, max_batch=B, k1_variant=args.variant | (args.timing_stride << 16),
                   flags=K.AGR_CFG_PERSISTENCE | K.AGR_CFG_TIMING | args.diag_flags | id_flags, id_secret=ID_SECRET)
    nanos0 = 1700000000000000000 + rank * 10_000_000_000        # each rank (shard) owns its own agent ids
    for k in range(wl["agents"]):
        eng.set_agent_state(A.synth_agent_id(k, agent_nanos0=nanos0), "running")
    synth = dict(seed=2 + rank, n_agents=wl["agents"], zipf_milli=wl["zipf_milli"], dup_permille=wl["dup_permille"], agent_nanos0=nanos0)
    first = eng.reserve_rows(B)
    for s in range(1, W + S):
        eng.reserve_rows(B)
    mint_base = first if id_flags else None                      # stream index j -> row first + j
    for s in range(W + S):                                       # records resident in HBM before the timed region
        eng.synth_fill_rows(s * B, first + s * B, B, mint_base=mint_base, **synth)
    stream = torch.cuda.ExternalStream(eng.stream(), device=torch.device("cuda", local_rank))
    sampler.wait_ready()
    for s in range(W):
        eng.ingest_rows_async(first + s * B, B)
    eng.sync()
    eng.kernel_time()                                            # drop warm-up launches from the kernel timer
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.mark()
    t0 = time.perf_counter()
    ev0.record(stream)
    for s in range(W, W + S):
        eng.ingest_rows_async(first + s * B, B)
    ev1.record(stream)
    eng.sync()
    torch.cuda.synchronize()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    sampler.unmark()
    if dist:
        dist.barrier()
    dev_ms = ev0.elapsed_time(ev1)
    k_ms, k_n = eng.kernel_time()
    clocks = sampler.stop()
    st = eng.stats()
    assert st["ingested"] == (W + S) * B, st
    if args.dump_outputs and rank == 0:
        dump_verdicts(args.dump_outputs, eng.debug_read("route", first + (W + S - 1) * B, B))
    if args.diag_flags:
        print("WARNING: diagnostic flags set; numbers below are for attribution only", file=sys.stderr)
    # ---- e2e through the public C-ABI call with pinned host buffers (H2D + kernels + D2H verdicts timed)
    # a two-slot pinned ring, like a host producer would use: the NEXT step's records are written while (here: before) the
    # current slot is ingested, so the slot being DMA'd is not sitting dirty in the host caches
    pins = [eng.pinned(B), eng.pinned(B)]
    pin_v = eng.pinned(B, A.verdict_dtype)
    pin_ids = eng.pinned(B * 16, np.uint8)
    ids_view = pin_ids.array.reshape(B, 16)
    e_times = []
    launches_before = st["k1_launches"]
    e_mint = (eng, first) if id_flags else None
    parallel_fill(A, pins[0].array, (W + S) * B, wl, synth["seed"], nanos0, mint=e_mint)
    for s in range(e_warm + e_steps):
        if s + 1 < e_warm + e_steps:
            parallel_fill(A, pins[(s + 1) % 2].array, (W + S + s + 1) * B, wl, synth["seed"], nanos0, mint=e_mint)
        if dist:
            dist.barrier()
        t = time.perf_counter()
        eng.ingest_ex(pins[s % 2].array, pin_v.array, ids_view)   # verdicts AND Request.IDs back on the host
        dt = time.perf_counter() - t
        verdicts = pin_v.array
        if s >= e_warm:
            e_times.append(dt)
    assert (verdicts["code"] != 0).all() and ids_view.any(axis=1).all()
    if id_flags:
        assert (ids_view[:64] == eng.mint_ids(eng.stats()["rows_used"] - B, 64)).all()
    del verdicts, ids_view
    pins[0].free(); pins[1].free(); pin_v.free(); pin_ids.free()
    e_ms = 1e3 * sum(e_times) / len(e_times)
    # ---- secondary kernels (SURVEY 8d): K2 over one batch of outcomes, K3 replay scan over the slab (device time)
    secondary = None
    if rank == 0 and not args.no_secondary:
        host = A.synth_fill_host(W * B, B, mint=(eng, first) if id_flags else None, **synth)   # the first timed batch
        outs = eng.pinned(B, A.outcome_dtype)
        outs.array["request_id"] = eng.mint_ids(first + W * B, B) if id_flags else host["request_id"]
        outs.array["agent_id"] = host["agent_id"]
        outs.array["kind"] = K.AGR_OUT_RESPONSE; outs.array["http_status"] = 200
        outs.array["seq"] = (W + S + 8) * B                          # processed_at: after every created_at of the run
        if wl["dup_permille"]:
            rep = (host["flags"] & 1) != 0
            outs.array["request_id"][rep] = host["replay_of"][rep]
        eng.complete(outs.array, want_results=False)
        k2_ms = eng.op_time(0)
        outs.free()
        # a tick where 1/16 of the agents are running with a backlog (every un-completed row is still pending)
        for k in range(wl["agents"]):
            if k % 16:
                eng.set_agent_state(A.synth_agent_id(k, agent_nanos0=nanos0), "stopped")
        disp, _ = eng.replay_scan(with_records=False, cap=1 << 22)
        k3_ms = eng.op_time(1)
        for k in range(wl["agents"]):
            eng.set_agent_state(A.synth_agent_id(k, agent_nanos0=nanos0), "running")
        scanned = eng.stats()["rows_used"]
        # K5: the JSON wire form (json.Marshal(requests.Request)) of the same batch, left on the device
        eng.rows_json(first + W * B, B, as_array=True, fetch=False)        # warm-up: sizes the output buffer
        json_bytes = eng.rows_json(first + W * B, B, as_array=True, fetch=False)
        k5_ms = eng.op_time(2)
        peak_s, _ = measured_peak()
        secondary = {"k2_complete": {"outcomes": B, "ms": k2_ms, "outcomes_per_s": B / (k2_ms * 1e-3), "launches": 3,
                                     "algorithmic_bytes_per_outcome": 72, "GBps": 72 * B / (k2_ms * 1e-3) / 1e9,
                                     "frac_of_peak": 72 * B / (k2_ms * 1e-3) / 1e9 / peak_s,
                                     "survey_bytes_per_outcome": 16, "frac_of_peak_survey_bytes": 16 * B / (k2_ms * 1e-3) / 1e9 / peak_s,
                                     "note": "72 B = the 64 B agr_outcome the ABI delivers (16 B id + 32 B agent id + kind/status/time) + 4 B state RMW + 4 B list append; SURVEY 8d sketched an 8 B descriptor (16 B/outcome)"},
                     "k3_replay_scan": {"rows_scanned": scanned, "dispatched": int(len(disp)), "ms": k3_ms,
                                        "rows_per_s": scanned / (k3_ms * 1e-3), "algorithmic_bytes_per_row": 8,
                                        "GBps": 8 * scanned / (k3_ms * 1e-3) / 1e9},
                     "k5_json": {"records": B, "ms": k5_ms, "records_per_s": B / (k5_ms * 1e-3), "json_bytes": json_bytes,
                                 "algorithmic_bytes_per_record": 512 + json_bytes / B,
                                 "GBps": (512 * B + json_bytes) / (k5_ms * 1e-3) / 1e9,
                                 "note": "measure + scan + emit kernels and the host's read of the total between them"}}
        eng_sust = measure_sustained(A, K, torch, local_rank, args.variant)
        secondary["sustained_ring"] = eng_sust
    # ---- the other named configurations, each on a fresh engine with its own roofline: the same workload in the OTHER id
    # mode ("mint" = the engine mints Request.ID like StoreRequest does, requests.go:87, ids are a keyed bijection of the row;
    # "hash" = caller-supplied random ids kept in the dedupe index: one CAS.128 + RED per stored record), and the other
    # single-GPU workload in both modes
    subs = []
    if not args.no_other_mode:
        o_steps = min(S, 20)
        other_wl = "c2" if args.workload == "c3" else "c3"
        for wname, mode in ((args.workload, "hash" if id_flags else "mint"), (other_wl, "mint"), (other_wl, "hash")):
            o_dev_ms, o_k = measure_resident(A, K, torch, dist, args, WORKLOADS[wname], rank, local_rank,
                                             K.AGR_CFG_MINT_IDS if mode == "mint" else 0, o_steps, W)
            subs.append((wname, mode, o_dev_ms / o_steps, o_k))
    # ---- N > 1: the exchange path (BASELINE config 4): 5 % of every rank's batch are replay-flagged records whose agent
    # lives on another shard -> K4 bin/pack, NCCL all-to-all to the owners, K1 there, verdicts back.  Host buffers in,
    # verdicts out, wall clock with a barrier on both sides (max over ranks by construction of the barrier).
    exchange = None
    if dist and not args.no_exchange:
        from agentainer_lab_b200.sharding import owned_agents, make_rank_batch
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)                     # NCCL prints its version banner to stdout on communicator creation
        try:
            uid = [A.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            eng.comm_init(uid[0], rank, world)
        finally:
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
        own = owned_agents(world, 64, nanos0=1800000000000000000)
        for a in own[rank]:
            eng.set_agent_state(a, "running")
        xn, x_times, sent, recvd = B // 4, [], 0, 0
        xpins = [eng.pinned(xn), eng.pinned(xn)]           # two-slot ring like the e2e leg: the slot being DMA'd is not dirty in the CPU caches
        xpins[0].array[:] = make_rank_batch(rank, world, own, xn, seed=50, p_cross_replay=0.05, first_index=0)
        for s in range(1 + args.x_steps):
            if s + 1 < 1 + args.x_steps:
                xpins[(s + 1) % 2].array[:] = make_rank_batch(rank, world, own, xn, seed=51 + s, p_cross_replay=0.05, first_index=(s + 1) * xn)
            dist.barrier()
            t = time.perf_counter()
            xv, info = eng.ingest_sharded(xpins[s % 2].array)
            dist.barrier()
            dt = time.perf_counter() - t
            if s >= 1:
                x_times.append(dt); sent += info.n_sent; recvd += info.n_received
        assert (xv["code"] == K.AGR_V_FORWARD).all()
        xpins[0].free(); xpins[1].free()
        x_ms = 1e3 * sum(x_times) / len(x_times)
        cnt = torch.tensor([sent, recvd], device="cuda", dtype=torch.float64)
        dist.all_reduce(cnt)
        exchange = {"value": world * xn / (x_ms * 1e-3), "unit": "requests/s", "records_per_step_per_gpu": xn,
                    "cross_shard_fraction": float(cnt[0]) / (world * xn * len(x_times)), "ms_per_step": x_ms,
                    "nvlink_bytes_per_step": float(cnt[0]) * (512 + 8) / len(x_times),
                    "api": "agr_ingest_sharded (pinned host records DMA'd straight into slab rows, K4 bins in place and packs only the cross-shard records, NCCL all-to-all, K1 at the owner, verdicts back)"}
        exchange["verified_against_oracle"] = verify_exchange(A, K, dist, rank, world, local_rank)
    if dist:
        t_all = torch.tensor([dev_ms, e_ms, k_ms / max(1, k_n)] + [x for sub in subs for x in sub[2:]], device="cuda", dtype=torch.float64)
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
        vals = [float(x) for x in t_all.tolist()]
        dev_ms, e_ms, k_avg = vals[:3]
        subs = [(sub[0], sub[1], vals[3 + 2 * i], vals[4 + 2 * i]) for i, sub in enumerate(subs)]
    else:
        k_avg = k_ms / max(1, k_n)
    if rank == 0:
        peak, peak_src = measured_peak()
        achieved = ALG_BYTES_PER_RECORD * B / (k_avg * 1e-3) / 1e9
        traffic_of = lambda mode: k1_traffic(mode, args.variant)
        traffic, traffic_src = traffic_of(args.id_mode)
        cpu = cpu_port_single(A, wl) if world == 1 and not args.no_cpu else None
        line = {
            "metric": METRIC, "value": world * B * S / (dev_ms * 1e-3), "unit": "requests/s", "n_gpus": world, "steps": S, "warmup": W,
            "ms_per_step": dev_ms / S, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic",
            "config": {"workload": wl["name"], "records_per_step_per_gpu": B, "agents_per_gpu": wl["agents"], "record_bytes": 512,
                       "parallelism": f"shard{world} by FNV-1a64(agent_id) mod {world}; fresh traffic steered to the owner (no collective); the exchange path is measured separately under \"exchange\"" if world > 1 else "single",
                       "l2": "each step reads a fresh 512 MiB batch (> 126 MB L2); no explicit flush",
                       "k1_variant": args.variant,
                       "id_mode": args.id_mode + (" (engine-minted Request.ID = keyed bijection of the row, as StoreRequest mints uuid.New(); no dedupe-index table)"
                                                   if id_flags else " (caller-supplied random ids in a 32 B/slot dedupe index)")},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": traffic_src,
                         "kernel": "k1_ingest", "kernel_ms": k_avg, "launches_timed": k_n, "launches_in_timed_region": S,
                         "timing": f"CUDA events on the engine's stream around the K1 kernel of every {max(1, args.timing_stride)}-th launch of the timed region (an event pair per launch costs the back-to-back loop ~5 us a step)" if args.timing_stride > 1 else "CUDA events on the engine's stream around the K1 kernel of every launch of the timed region",
                         "algorithmic_bytes_per_record": ALG_BYTES_PER_RECORD, "peak_source": peak_src},
            "e2e": {"value": world * B / (e_ms * 1e-3), "unit": "requests/s", "h2d_bytes_per_step": B * 512, "d2h_bytes_per_step": B * 24,
                    "steps": len(e_times), "ms_per_step": e_ms, "api": "agr_ingest_ex (pinned host records in; verdicts + Request.IDs out)",
                    "host_cpus_local_to_gpu": local_cpus},
            "gpu_launches": S * 2, "wall_ms_timed_region": wall_ms, "device_ms_timed_region": dev_ms, "clocks": clocks,
        }
        if cpu:
            line["cpu_baseline"] = cpu
        if exchange:
            line["exchange"] = exchange
        if secondary:
            line["secondary_kernels"] = secondary
        if subs:
            cfgs = {}
            for wname, mode, ms, kms in subs:
                ach = ALG_BYTES_PER_RECORD * B / (kms * 1e-3) / 1e9
                tr, tr_src = traffic_of(mode)
                cfgs[f"{wname}_{mode}"] = {"workload": WORKLOADS[wname]["name"], "id_mode": mode, "value": world * B / (ms * 1e-3), "unit": "requests/s",
                                           "ms_per_step": ms, "steps": min(S, 20),
                                           "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                                        "kernel": "k1_ingest", "kernel_ms": kms, "traffic": tr, "traffic_source": tr_src}}
            line["configs"] = cfgs
    eng.close()
    if rank == 0:
        if world == 1 and not args.no_callers:
            line["e2e_callers"] = run_callers(local_rank)
        print(json.dumps(line))
    if dist:
        dist.destroy_process_group()


def make_var_blob(A, n, first_index, seed, n_agents, nanos0, rng):
    """n variable-length records (BASELINE config 5): the synthetic 512 B stream's headers / paths / HTTP headers with
    bodies of log-uniform length in [128 B, 4 KB]."""
    fixed = A.synth_fill_host(first_index, n, seed=seed, n_agents=n_agents, agent_nanos0=nanos0)
    body = np.exp(rng.uniform(np.log(128), np.log(4096), n)).astype(np.int64)
    ph = fixed["path_len"].astype(np.int64) + fixed["hdr_len"]
    lens = 96 + ((ph + body + 15) // 16) * 16
    offs = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lens, out=offs[1:])
    blob = rng.integers(32, 127, int(offs[-1]), dtype=np.uint8)
    fixed["body_len"] = body
    raw = fixed.view(np.uint8).reshape(n, 512)
    cols = np.arange(96 + 92)                                   # header + path + HTTP headers (92 B in the synthetic stream)
    blob[(offs[:-1, None] + cols[None, :]).ravel()] = raw[:, :188].ravel()
    return blob, offs.astype(np.uint32), int(offs[-1])


def run_c5(args, rank, world, local_rank):
    """--workload c5 (BASELINE configs[4]): a SUSTAINED stream of variable-length records (bodies log-uniform in 128 B .. 4 KB)
    through a ring-mode engine on every GPU, with the whole state machine in the loop:
      every batch   agr_ingest_var (byte-tiled K1v, 1-D bulk TMA)  ->  agr_complete for every forwarded request (K2)
                    ->  agr_expire + agr_reclaim (TTL sweep, rows / bytes back to the ring);
      every 25th    1 % of the agents CRASH for that batch: their container is dead while their status still says running, so
                    the proxy forwards, the dial fails (AGR_OUT_DIAL_ERR, Q12) and the records stay pending; then they restart,
                    one ReplayWorker tick (agr_replay_scan_var, K3) hands back their FULL pending queues, every record is
                    re-injected replay-flagged (K1v: dedupe hit on the stored id) and completed TWICE (server side + worker
                    side, Q7).
    Shards are independent (agents steered to their owner): weak scaling, no data-path collective.  value = records / K1v kernel
    time (there is no resident-input form of the variable-length ingest); e2e = records / wall time of the WHOLE loop."""
    import torch
    import agentainer_lab_b200 as A
    from agentainer_lab_b200 import constants as K
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        init_nccl_quietly(dist, torch, local_rank)
    local_cpus = bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    n, na, W = 1 << 18, 256, max(3, args.warmup)
    total_target = 100_000_000 if world == 8 else 6_000_000 * world
    S = args.steps if args.steps is not None else -(-total_target // (world * n))
    R = 8 * n
    TTLB = 4                                                           # a record lives four batches
    rng = np.random.default_rng(7 + rank)
    nanos0 = 1700000000000000000 + rank * 10_000_000_000
    eng = A.Engine(device=local_rank, slab_rows=R, max_agents=1024, max_batch=n, vslab_bytes=R * 1500, k1_variant=args.variant, log_entries=4 * R,
                   flags=K.AGR_CFG_PERSISTENCE | K.AGR_CFG_VARLEN | K.AGR_CFG_MINT_IDS | K.AGR_CFG_TIMING | K.AGR_CFG_RING)
    names = [A.synth_agent_id(k, agent_nanos0=nanos0) for k in range(na)]
    eng.set_agent_states(names, ["running"] * na)
    names_b = np.array([x.encode() for x in names], dtype="S32")
    # four distinct pinned blobs, cycled; created_at (seq) is patched per use so the TTL clock keeps running
    blobs = []
    for q in range(4):
        blob, offs, nbytes = make_var_blob(A, n, q * n, 5 + rank, na, nanos0, rng)
        pin = eng.pinned(nbytes, np.uint8); pin.array[:] = blob
        hdr_idx = (offs[:-1, None].astype(np.int64) + np.arange(96)[None, :]).ravel()
        agents = blob[hdr_idx].reshape(n, 96)[:, 32:64].copy().view("S32").ravel()
        tmpl = eng.pinned(n, A.outcome_dtype)                           # the batch's outcomes, agent ids and kinds filled in once
        tmpl.array["agent_id"] = agents; tmpl.array["kind"] = K.AGR_OUT_RESPONSE; tmpl.array["http_status"] = 200
        blobs.append((pin, offs, nbytes, agents, (offs[:-1].astype(np.int64) + 64) // 8, tmpl))
    arange_n = np.arange(n, dtype=np.uint64)
    def patch_seq(pin, seq_word, first_seq):                             # created_at is 8-byte aligned: one scatter of n words
        pin.array.view(np.uint64)[seq_word] = first_seq + arange_n
    stats = dict(records=0, bytes=0, dial=0, replayed=0, crash_cycles=0, completions=0)
    wall = []
    def step(b, timed):
        pin, offs, nbytes, agents, seq_off, tmpl = blobs[b % 4]
        patch_seq(pin, seq_off, b * n)
        crash = (b % 25 == 24)
        dead = names_b[rng.choice(na, max(1, na // 100), replace=False)] if crash else None
        t0 = time.perf_counter()
        v, ids, _ = eng.ingest_var(pin.array, offs)
        o = tmpl.array
        o["request_id"] = ids; o["seq"] = b * n + n
        n_dial = 0
        if crash:
            hit = np.isin(agents, dead)
            o["kind"][hit] = K.AGR_OUT_DIAL_ERR                          # "dial tcp ... connection refused": stays pending (server.go:600-605)
            n_dial = int(hit.sum())
        eng.complete(o, want_results=False)
        if crash:
            o["kind"][hit] = K.AGR_OUT_RESPONSE
        n_rep = 0
        if crash:
            # the agents are back: one tick replays their whole pending queues in arrival order
            disp, rblob, roffs = eng.replay_scan_var(cap=1 << 16, blob_cap=1 << 27)
            n_rep = len(disp)
            assert n_rep == n_dial, (n_rep, n_dial)
            if n_rep:
                ro = roffs.astype(np.int64)
                rb = np.ascontiguousarray(rblob)
                fl = (ro[:-1, None] + 72 + np.arange(4)[None, :]).ravel()
                flags = rb[fl].view(np.uint32) | 1                        # X-Agentainer-Replay: true
                rb[fl] = flags.view(np.uint8)
                rb[(ro[:-1, None] + 16 + np.arange(16)[None, :]).ravel()] = disp["request_id"].reshape(-1)   # X-Agentainer-Request-ID
                rv, _, _ = eng.ingest_var(rb, ro.astype(np.uint32))
                assert (rv["code"] == K.AGR_V_FORWARD).all() and ((rv["flags"] & K.AGR_VF_KNOWN) != 0).all()
                ragents = rb[(ro[:-1, None] + 32 + np.arange(32)[None, :]).ravel()].reshape(n_rep, 32).copy().view("S32").ravel()
                ro2 = np.zeros(2 * n_rep, dtype=A.outcome_dtype)          # interceptTransport's StoreResponse, then the worker's (Q7)
                ro2["request_id"] = np.repeat(disp["request_id"], 2, axis=0); ro2["agent_id"] = np.repeat(ragents, 2)
                ro2["kind"] = K.AGR_OUT_RESPONSE; ro2["http_status"] = 200; ro2["seq"] = b * n + n + 1
                eng.complete(ro2, want_results=False)
        eng.expire((b + 1) * n, TTLB * n, want_count=False)
        eng.reclaim_async()
        dt = time.perf_counter() - t0
        assert (v["code"] == K.AGR_V_FORWARD).all()
        if timed:
            wall.append(dt)
            stats["records"] += n; stats["bytes"] += nbytes; stats["dial"] += n_dial; stats["replayed"] += n_rep
            stats["crash_cycles"] += 1 if crash else 0; stats["completions"] += n - n_dial + 2 * n_rep
    for b in range(W):
        step(b, False)
    eng.kernel_time()
    st0 = eng.stats()
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    t_all0 = time.perf_counter()
    for b in range(W, W + S):
        step(b, True)
    torch.cuda.synchronize()
    loop_s = time.perf_counter() - t_all0
    if dist:
        dist.barrier()
    k_ms, k_n = eng.kernel_time()
    st = eng.stats()
    # size-independent properties of the whole run: every fresh record stored, every replay a dedupe hit, every forwarded
    # request completed exactly once (replayed ones twice more), nothing left pending, the ring never over-full
    assert st["stored"] - st0["stored"] == stats["records"], (st, stats)
    assert st["dedupe_hits"] - st0["dedupe_hits"] == stats["replayed"] and st["dial_errors"] - st0["dial_errors"] == stats["dial"], (st, stats)
    assert st["completions"] - st0["completions"] == stats["completions"], (st, stats)
    assert st["rows_used"] - st["rows_tail"] <= R
    pend = sum(len(eng.list(a, K.AGR_LIST_PENDING, cap=1 << 16)) for a in names[:: max(1, na // 16)])
    assert pend == 0, pend
    eng.close()
    vals = torch.tensor([loop_s, k_ms, float(stats["records"]), float(stats["bytes"]), float(stats["replayed"]), float(stats["crash_cycles"])],
                        dtype=torch.float64, device="cuda" if dist else "cpu")
    mx = vals.clone(); sm = vals.clone(); per_gpu = [stats["records"]]
    if dist:
        dist.all_reduce(mx, op=dist.ReduceOp.MAX); dist.all_reduce(sm)
        g = [None] * world
        dist.all_gather_object(g, stats["records"]); per_gpu = g
    if rank == 0:
        loop_s, k_ms = float(mx[0]), float(mx[1])
        recs, nbytes, replayed, cycles = float(sm[2]), float(sm[3]), float(sm[4]), float(sm[5])
        peak, peak_src = measured_peak()
        alg = (nbytes + 8 * recs) / world                                # per GPU; the replayed records' re-reads are not counted
        ach = alg / (k_ms * 1e-3) / 1e9
        line = {"metric": METRIC.replace("512B", "128B-4KB"), "value": recs / (k_ms * 1e-3), "unit": "requests/s", "n_gpus": world, "steps": S, "warmup": W,
                "ms_per_step": k_ms / max(1, S), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
                "config": {"workload": f"C5: {world} x B200, {int(recs)} records sustained through a ring ({R} rows, {R * 1500 >> 20} MiB of bytes per GPU), bodies log-uniform in [128 B, 4 KB], every 25th batch 1% of the agents crash (dial errors -> pending) then restart + tick + full pending-queue replay",
                           "records_per_step_per_gpu": n, "mean_record_bytes": nbytes / recs, "agents_per_gpu": na, "per_gpu_records": per_gpu,
                           "parallelism": f"shard{world}: agents steered to their owner, no data-path collective" if world > 1 else "single",
                           "l2": "each step reads a fresh ~170 MiB blob (> 126 MB L2)",
                           "value_is": "records / K1v kernel time (CUDA events around the kernel, summed); e2e is the whole loop"},
                "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                             "kernel": "k1v_tile_index + k1_ingest_var", "kernel_ms": k_ms / max(1, k_n), "launches_timed": k_n,
                             "algorithmic_bytes": "stored record length + 8 per record (SURVEY 8d)", "peak_source": peak_src},
                "e2e": {"value": recs / loop_s, "unit": "requests/s", "h2d_bytes_per_step": nbytes / world / S + n * 64, "d2h_bytes_per_step": n * 24,
                        "ms_per_step": 1e3 * loop_s / S, "api": "agr_ingest_var + agr_complete + agr_expire + agr_reclaim every batch; agr_replay_scan_var + replay-flagged re-ingest + double completion on crash cycles",
                        "host_cpus_local_to_gpu": local_cpus},
                "crash_replay": {"cycles": int(cycles), "records_replayed": int(replayed), "agents_crashed_per_cycle": max(1, na // 100)},
                "gpu_launches": int(S * 12)}
        print(json.dumps(line))
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 200; c4: 10; c5: enough batches for its record target)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS) + ["c4", "c5"])
    ap.add_argument("--variant", type=lambda x: int(x, 0), default=0)
    ap.add_argument("--timing-stride", type=int, default=8, help="CUDA events around the K1 kernel of every k-th launch of the timed region (1 = every launch)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-exchange", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-other-mode", action="store_true")
    ap.add_argument("--no-callers", action="store_true")
    ap.add_argument("--id-mode", default="mint", choices=["mint", "hash"])
    ap.add_argument("--x-steps", type=int, default=3)
    ap.add_argument("--diag-flags", type=lambda x: int(x, 0), default=0, help="extra AGR_CFG_DIAG_* bits (results invalid; attribution only)")
    ap.add_argument("--rows", type=int, default=0, help="override slab rows (table size follows)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="c2 / c3: write the verdicts of the last timed step to DIR/verdict_<field>.npy (float64)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload not in WORKLOADS):
        ap.error("--dump-outputs covers the GPU path of the c2 / c3 workloads")
    if args.steps is None and (args.impl == "reference" or args.workload in WORKLOADS):
        args.steps = 200
    args.warmup = max(3, args.warmup) if args.impl == "ours" else args.warmup
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        # the CPU path does the same per-record work whatever the GPU-side sharding: c4 / c5 are timed on their 512 B base stream
        return run_reference(args, WORKLOADS.get(args.workload, WORKLOADS["c2"]), rank, world)
    if args.workload == "c5":
        return run_c5(args, rank, world, local_rank)
    if args.workload == "c4":
        return run_c4(args, rank, world, local_rank)
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl, rank, world)
    else:
        run_ours(args, wl, rank, world, local_rank)


if __name__ == "__main__":
    main()
