"""The single-request front end for VARIABLE-LENGTH records (AGR_CFG_VARLEN | AGR_CFG_COMBINE): agr_ingest_var / agr_complete
with n <= 32 and agr_submit_ingest_var go through the pinned request ring (a record of stored length L takes ceil(L / 512)
consecutive slots), the dispatcher and the resident service kernel.  Oracle parity, the same engine state as the batch path,
threads over several laps of the ring, the byte ring, a full byte slab, and tickets held beyond the ring's capacity."""
import ctypes
import json
import os
import subprocess
import threading

import numpy as np
import pytest

import agentainer_lab_b200 as A
from agentainer_lab_b200 import constants as K
from kats import SCENARIOS, load_golden
from scenario import Req, rid_of, make_var_batch, run_oracle, run_engine, assert_same, random_scenario
from test_varlen_gpu import with_bodies

pytestmark = pytest.mark.gpu
GOLD, _ = load_golden()
VAR = K.AGR_CFG_PERSISTENCE | K.AGR_CFG_VARLEN
SVC = VAR | K.AGR_CFG_COMBINE


def engine(flags=SVC, **kw):
    kw.setdefault("slab_rows", 1 << 15)
    kw.setdefault("max_agents", 256)
    kw.setdefault("vslab_bytes", 256 << 20)
    return A.Engine(flags=flags, **kw)


def outcome(rid, agent, kind, http=200, seq=7):
    o = np.zeros(1, dtype=A.outcome_dtype)
    o["request_id"], o["agent_id"], o["kind"], o["http_status"], o["seq"] = np.frombuffer(rid, dtype=np.uint8), agent.encode(), kind, http, seq
    return o


def cksum(rec: np.ndarray) -> int:
    w = rec.view(np.uint32).astype(np.uint64)
    c0 = int(w.sum()) & 0xFFFFFFFF
    c1 = int((w * np.arange(1, len(w) + 1, dtype=np.uint64)).sum()) & 0xFFFFFFFF
    return (c1 << 32) | c0


@pytest.mark.parametrize("kat", sorted(SCENARIOS))
@pytest.mark.parametrize("flags", [SVC, SVC | K.AGR_CFG_MINT_IDS])
def test_kats_through_the_ring(kat, flags):
    ev = with_bodies(SCENARIOS[kat], 1)
    with engine(flags) as eng:
        got = run_engine(eng, ev, max_batch=32)
        assert eng.stats()["svc_ops"] > 0
    exp = GOLD[kat]
    assert got.verdicts == exp["verdicts"] and got.ticks == exp["ticks"] and got.records == exp["records"]
    for a, qs in exp["lists"].items():
        assert got.lists[a] == qs, (kat, a)


@pytest.mark.parametrize("seed", range(4))
def test_random_streams_through_the_ring(seed):
    ev = with_bodies(random_scenario(400 + seed, n_events=500, n_agents=2 + seed % 4, p_replay=0.15), seed)
    with engine(SVC | (K.AGR_CFG_MINT_IDS if seed % 2 else 0)) as eng:
        got = run_engine(eng, ev, max_batch=32, rng=np.random.default_rng(seed))
        s = eng.stats()
    assert_same(run_oracle(ev), got)
    assert s["svc_ops"] >= s["stored"] > 0


def _state(eng, n):
    return {w: eng.debug_read(w, 0, n).tolist() for w in ("state", "route", "aux", "cksum")}


@pytest.mark.parametrize("flags", [VAR, VAR | K.AGR_CFG_MINT_IDS])
def test_single_requests_leave_the_state_of_the_batch_path(flags, tmp_path):
    """One stream, two append-only engines: agr_ingest_var batches vs one record per call through the ring (and outcomes of up
    to 32 per call through it as well).  Rows, row words, stored bytes, the JSON wire form and agr_verify agree; a snapshot /
    restore of the ring engine changes none of it.  (Engine-minted ids: one id secret for both, and no replay-flagged requests —
    a replay names its original by the id the engine minted, which the batch caller does not know yet when both are in one batch.)"""
    mint = bool(flags & K.AGR_CFG_MINT_IDS)
    ev = with_bodies(random_scenario(77, n_events=600, n_agents=4, p_replay=0.0 if mint else 0.1), 5)
    with engine(flags, id_secret=0x5EC2E7) as ref, engine(flags | K.AGR_CFG_COMBINE, id_secret=0x5EC2E7) as eng:
        o1 = run_engine(ref, ev)
        o2 = run_engine(eng, ev, max_batch=1)
        assert_same(o1, o2)
        n = ref.stats()["rows_used"]
        assert eng.stats()["rows_used"] == n and eng.stats()["svc_ops"] >= n > 100
        want = _state(ref, n)
        js = ref.rows_json(0, n)[0]
        recs = {}
        for e in ev:
            if e[0] == "req" and not e[1].replay:
                recs[(e[1].agent_id, e[1].rid)] = ref.get_record_var(e[1].agent_id, e[1].rid) if not (flags & K.AGR_CFG_MINT_IDS) else None
        snap = str(tmp_path / "svc_var.snap")
        eng.snapshot(snap)
        for e2 in (eng, A.Engine(flags=flags | K.AGR_CFG_COMBINE, slab_rows=1 << 15, max_agents=256, vslab_bytes=256 << 20, id_secret=0x5EC2E7,
                                 restore_from=snap)):
            assert _state(e2, n) == want
            assert e2.rows_json(0, n)[0] == js
            assert e2.verify()[1] == 0
            for (a, rid), raw in recs.items():
                got = e2.get_record_var(a, rid)
                assert (raw is None) == (got is None) and (raw is None or raw.tobytes() == got.tobytes())
            if e2 is not eng:
                e2.close()


def test_single_request_var_under_threads():
    """32 threads of blocking single-request calls (agr_ingest_var n = 1, then agr_complete n = 1 for the forwarded ones) with
    records of 96 B .. 8192 B: enough slots to lap the 16384-slot ring more than three times, so runs cross its end."""
    nt, per = 32, 240
    agents = ["agent-%d" % k for k in range(4)]
    rng = np.random.default_rng(9)
    bodies = {}
    for t in range(nt):
        for i in range(per):
            m = (t + i) % 3
            bodies[(t, i)] = b"" if m == 0 else (bytes(rng.integers(32, 127, 8192 - 96 - len(f"/agent/{agents[(t + i) % 4]}/c"), dtype=np.uint8)) if m == 1
                                                 else bytes(rng.integers(32, 127, int(np.exp(rng.uniform(np.log(128), np.log(4096)))), dtype=np.uint8)))
    with engine(SVC | K.AGR_CFG_MINT_IDS, slab_rows=1 << 15, max_agents=8) as eng:
        for k, a in enumerate(agents):
            eng.set_agent_state(a, "stopped" if k % 2 else "running")
        results = [[] for _ in range(nt)]
        errors = []

        def worker(t):
            try:
                for i in range(per):
                    a = agents[(t + i) % 4]
                    blob, offs = make_var_batch([Req(a, rid_of(1 + t * per + i), 1 + t * per + i, subpath="/c", body=bodies[(t, i)], headers={})])
                    v, ids, first = eng.ingest_var(blob, offs)
                    kind = None
                    if int(v[0]["code"]) == K.AGR_V_FORWARD:
                        kind = K.AGR_OUT_ERROR if (t + i) % 5 == 0 else K.AGR_OUT_RESPONSE
                        assert list(eng.complete(outcome(bytes(ids[0]), a, kind))) == [0]
                    results[t].append((a, int(v[0]["code"]), first, bytes(ids[0]), kind, blob))
            except Exception as e:                                               # noqa: BLE001
                errors.append(repr(e))

        ths = [threading.Thread(target=worker, args=(t,)) for t in range(nt)]
        for th in ths:
            th.start()
        for th in ths:
            th.join()
        assert not errors, errors[:3]
        flat = [x for r in results for x in r]
        lens = [len(x[5]) for x in flat]
        assert min(lens) == 112 and max(lens) == 8192                         # (header + the shortest path: 96 B is the ticket test's)
        slots = sum((n + 511) // 512 for n in lens) + sum(1 for x in flat if x[4] is not None)
        assert slots > 3 * A.load_library().agr_ring_capacity()
        assert len({x[2] for x in flat}) == nt * per                           # every request got its own row
        assert all((code == K.AGR_V_QUEUED) == (agents.index(a) % 2 == 1) for a, code, _, _, _, _ in flat)
        assert all(bytes(eng.mint_ids(first, 1)[0]) == rid for _, _, first, rid, _, _ in flat)
        for k, a in enumerate(agents):
            mine = sorted((first, rid, kind) for aa, _, first, rid, kind, _ in flat if aa == a)
            pend = [bytes(x) for x in eng.list(a, K.AGR_LIST_PENDING, cap=1 << 14)]
            comp = [bytes(x) for x in eng.list(a, K.AGR_LIST_COMPLETED, cap=1 << 14)]
            if k % 2:
                assert pend == [rid for _, rid, _ in mine] and comp == []       # FIFO == row order
            else:
                assert pend == [rid for _, rid, kind in mine if kind == K.AGR_OUT_ERROR]
                assert sorted(comp) == sorted(rid for _, rid, kind in mine if kind == K.AGR_OUT_RESPONSE)
        ck = eng.debug_read("cksum", 0, nt * per)
        for a, _, first, rid, kind, blob in flat[::7]:
            raw = eng.get_record_var(a, rid)
            assert len(raw) == len(blob) and raw[96:].tobytes() == blob[96:].tobytes() and raw[16:80].tobytes() == blob[16:80].tobytes()
            st = (K.AGR_ST_PENDING, 1) if kind == K.AGR_OUT_ERROR else ((K.AGR_ST_COMPLETED, 0) if kind else (K.AGR_ST_PENDING, 0))
            assert (int(raw[84]), int(raw[85])) == st
            assert int(ck[first]) == cksum(blob)                              # the ingested bytes (the id as the caller sent it)
        assert eng.verify()[1] == 0
        s = eng.stats()
        assert s["stored"] == nt * per and 0 < s["svc_batches"] <= s["svc_ops"]


def test_byte_ring_fed_by_single_requests():
    """VARLEN | RING | COMBINE fed only by single requests: several laps of the byte ring with agr_expire + agr_reclaim between
    steps; live ids resolve, released ones do not."""
    R, per, ttl, vbytes = 4096, 128, 3 * 128, 2 << 20
    agent = "agent-1700000000000000001"
    rng = np.random.default_rng(4)
    with engine(SVC | K.AGR_CFG_MINT_IDS | K.AGR_CFG_RING, slab_rows=R, max_agents=4, max_batch=per, vslab_bytes=vbytes) as eng:
        eng.set_agent_state(agent, "stopped")
        ids_by_step, total = [], 0
        for step in range(60):
            ids = []
            for i in range(per):
                body = bytes(rng.integers(32, 127, int(np.exp(rng.uniform(np.log(128), np.log(4096)))), dtype=np.uint8))
                r = Req(agent, rid_of(1 + step * per + i), step * per + i, subpath="/c", body=body)      # seq = created_at
                blob, offs = make_var_batch([r])
                v, vid, _ = eng.ingest_var(blob, offs)
                assert int(v[0]["code"]) == K.AGR_V_QUEUED
                ids.append(bytes(vid[0])); total += len(blob)
            ids_by_step.append(ids)
            eng.expire((step + 1) * per, ttl)
            eng.reclaim()
            st = eng.stats()
            assert st["rows_used"] - st["rows_tail"] <= R
        assert total > 3 * vbytes and eng.stats()["rows_used"] > R
        assert eng.get_record_var(agent, ids_by_step[-1][5]) is not None
        assert eng.get_record_var(agent, ids_by_step[10][5]) is None
        assert eng.verify()[1] == 0


@pytest.mark.parametrize("ring", [False, True])
def test_full_byte_slab_answers_enospc(ring):
    agent = "agent-1"
    flags = SVC | K.AGR_CFG_MINT_IDS | (K.AGR_CFG_RING if ring else 0)
    with engine(flags, slab_rows=1 << 12, max_agents=4, max_batch=256, vslab_bytes=256 << 10) as eng:
        eng.set_agent_state(agent, "running")
        big = Req(agent, rid_of(1), 1, subpath="/c", body=bytes(8192 - 96 - len("/agent/agent-1/c")), headers={})
        ok = 0
        with pytest.raises(A.AgrError) as ei:
            for i in range(100):
                blob, offs = make_var_batch([big])
                eng.ingest_var(blob, offs)
                ok += 1
        assert ei.value.code == K.AGR_ENOSPC and 0 < ok <= 32
        blob, offs = make_var_batch([big])
        with pytest.raises(A.AgrError) as ei:
            eng.ingest_var(blob, offs)                              # still full, still answered
        assert ei.value.code == K.AGR_ENOSPC
        assert eng.stats()["stored"] == ok
        first = eng.list(agent, K.AGR_LIST_PENDING)[0]
        assert list(eng.complete(outcome(bytes(first), agent, K.AGR_OUT_RESPONSE))) == [0]   # outcomes still go through


def test_tickets_and_argument_checks():
    lib = A.load_library()
    with engine(SVC, slab_rows=1 << 12, max_agents=4) as eng:
        eng.set_agent_state("agent-1", "running")
        blobs = [make_var_batch([Req("agent-1", rid_of(i + 1), i + 1, subpath="/c", body=b"x" * (100 * i))])[0] for i in range(40)]
        tickets = [eng.submit_ingest_var(b) for b in blobs]
        assert None not in tickets
        got = [eng.poll(t, wait=True) for t in tickets]
        assert [g[1] for g in got] == [rid_of(i + 1) for i in range(40)] and all(g[3] == 0 for g in got)
        assert sorted(g[2] for g in got) == list(range(40))
        for i in (0, 13, 39):
            assert eng.get_record_var("agent-1", rid_of(i + 1)).tobytes()[96:] == blobs[i].tobytes()[96:]
        # a 96 B record (header only) whose header claims a payload: decided as AGR_VF_BAD_LEN, like the batch call does
        short = blobs[1][:96].copy()
        short[:16] = np.frombuffer(rid_of(1000), dtype=np.uint8)
        v, _, _, res = eng.poll(eng.submit_ingest_var(short), wait=True)
        assert res == 0 and int(v["flags"]) & K.AGR_VF_BAD_LEN
        sv, _, _ = eng.ingest_var(short, np.array([0, 96], dtype=np.uint32))
        assert int(sv[0]["flags"]) & K.AGR_VF_BAD_LEN
        bad = blobs[3][:-8].copy()
        with pytest.raises(A.AgrError):
            eng.submit_ingest_var(bad)                             # not a multiple of 16
        with pytest.raises(A.AgrError):
            eng.submit_ingest_var(np.zeros(8192 + 16, dtype=np.uint8))   # longer than AGR_VAR_MAX_RECORD
        t = np.zeros(1, dtype=np.uint64)
        rec = np.zeros(1, dtype=A.record_dtype)
        rc = lib.agr_submit_ingest(eng.h, ctypes.c_void_p(rec.ctypes.data), ctypes.c_void_p(t.ctypes.data))
        assert rc == K.AGR_EINVAL                                  # fixed-stride call, VARLEN engine
    with A.Engine(slab_rows=1 << 12, max_agents=4, flags=K.AGR_CFG_PERSISTENCE | K.AGR_CFG_COMBINE) as fx:
        with pytest.raises(A.AgrError):
            fx.submit_ingest_var(blobs[0])                         # variable-length call, fixed-stride engine


def test_more_var_tickets_held_than_ring_slots_never_deadlocks():
    """bench_callers with variable-length records: 8 threads x 4096 tickets in flight, each record 1 .. 9 slots, against 16384
    slots.  The run ends without errors."""
    exe = os.path.join(os.path.dirname(A.build_host()), "bench_callers")
    for threads, inflight in ((8, 4096), (8, 512), (16, 0)):
        res = subprocess.run([exe, str(threads), "1.0", "0", "mint", "64", str(inflight), "var"], capture_output=True, text=True, timeout=180)
        assert res.returncode == 0, (threads, inflight, res.stdout[-400:], res.stderr[-400:])
        d = json.loads(res.stdout.strip().splitlines()[-1])
        assert d["errors"] == 0 and d["round_trips"] > 0 and d["records"] == "var", d
