"""ctypes mirror of include/agentainer_gpu.h.  Test / bench harness only: the reference-facing boundary is the
C-ABI itself (a Go host binds it with cgo, see INTEGRATION.md).  Method names follow the ABI one to one."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Tuple

import numpy as np

from . import constants as K
from .build import build_native, lib_path

record_dtype = np.dtype([
    ("request_id", "u1", 16), ("replay_of", "u1", 16), ("agent_id", "S32"), ("seq", "<u8"), ("flags", "<u4"),
    ("path_len", "<u2"), ("hdr_len", "<u2"), ("body_len", "<u4"), ("status", "u1"), ("retry_count", "u1"),
    ("max_retries", "u1"), ("error_code", "u1"), ("resp_status", "<u2"), ("reserved0", "<u2"), ("reserved1", "<u4"),
    ("payload", "u1", 416)])
header_dtype = np.dtype([(n, record_dtype.fields[n][0]) for n in record_dtype.names if n != "payload"])   # the 96 B header
assert header_dtype.itemsize == 96
outcome_dtype = np.dtype([
    ("request_id", "u1", 16), ("agent_id", "S32"), ("kind", "u1"), ("reserved0", "u1"), ("http_status", "<u2"),
    ("reserved1", "<u4"), ("seq", "<u8")])
verdict_dtype = np.dtype([("code", "u1"), ("flags", "u1"), ("http_status", "<u2"), ("agent_slot", "<u4")])
dispatch_dtype = np.dtype([("rid", "<u8"), ("agent_slot", "<u4"), ("reserved", "<u4"), ("request_id", "u1", 16)])
assert record_dtype.itemsize == 512 and outcome_dtype.itemsize == 64
assert verdict_dtype.itemsize == 8 and dispatch_dtype.itemsize == 32


class AgrConfig(C.Structure):
    _fields_ = [("device", C.c_int32), ("flags", C.c_uint32), ("slab_rows", C.c_uint64), ("table_slots", C.c_uint64),
                ("max_agents", C.c_uint32), ("max_batch", C.c_uint32), ("log_entries", C.c_uint64),
                ("id_secret", C.c_uint64), ("vslab_bytes", C.c_uint64), ("resp_bytes", C.c_uint64),
                ("k1_variant", C.c_uint32), ("reserved", C.c_uint32)]


class AgrStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "rows_used", "rows_cap", "ingested", "stored", "replay_flagged", "dedupe_hits", "forwarded", "queued",
        "unavailable", "not_found", "dup_ids", "completions", "completion_misses", "failures", "dead_lettered",
        "dial_errors", "replay_scans", "replay_dispatched", "completed_log_len", "failed_log_len",
        "k1_launches", "k2_launches", "k3_launches", "k4_launches", "k5_launches", "rows_tail", "malformed", "log_overflow",
        "svc_batches", "svc_ops")] + [("agents", C.c_uint32), ("device", C.c_uint32)]


class AgrDecoded(C.Structure):
    _fields_ = [("status", C.c_uint8), ("retry_count", C.c_uint8), ("max_retries", C.c_uint8), ("has_response", C.c_uint8),
                ("resp_status", C.c_uint16), ("reserved", C.c_uint16), ("record_len", C.c_uint32), ("resp_hdr_len", C.c_uint32),
                ("resp_body_len", C.c_uint32), ("error_len", C.c_uint32), ("reserved2", C.c_uint32),
                ("created_at", C.c_uint64), ("processed_at", C.c_uint64), ("received_at", C.c_uint64)]


class AgrExchangeInfo(C.Structure):
    _fields_ = [("world", C.c_uint32), ("rank", C.c_uint32), ("n_local", C.c_uint32), ("n_sent", C.c_uint32),
                ("n_received", C.c_uint32), ("sent_to", C.c_uint32 * 32), ("received_from", C.c_uint32 * 32),
                ("first_rid", C.c_uint64), ("recv_first_rid", C.c_uint64)]


class AgrSynth(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("n_agents", C.c_uint32), ("zipf_milli", C.c_uint32),
                ("dup_permille", C.c_uint32), ("mint", C.c_uint32), ("agent_nanos0", C.c_uint64),
                ("mint_base_rid", C.c_uint64), ("mint_secret", C.c_uint64), ("mint_shard", C.c_uint32), ("mint_gen", C.c_uint32)]


class AgrResult(C.Structure):
    """agr_result: what agr_poll / agr_wait hand back for a ticket"""
    _fields_ = [("verdict", C.c_uint8 * 8), ("request_id", C.c_uint8 * 16), ("rid", C.c_uint64), ("result", C.c_int32), ("is_outcome", C.c_uint32)]


# every symbol include/agentainer_gpu.h declares (tests/test_abi.py cross-checks this list against the header)
ABI_SYMBOLS = [
    "agr_create", "agr_destroy", "agr_abi_version", "agr_last_error", "agr_strerror",
    "agr_set_agent_state", "agr_drop_agent", "agr_agent_slot",
    "agr_ingest", "agr_ingest_ex", "agr_ingest_var", "agr_replay_scan_var", "agr_get_record_var", "agr_complete", "agr_replay_scan", "agr_pending", "agr_get_record", "agr_list", "agr_stats_get",
    "agr_host_alloc", "agr_host_free", "agr_mint_ids", "agr_reserve_rows", "agr_ingest_rows", "agr_ingest_rows_async", "agr_sync",
    "agr_stream", "agr_kernel_time", "agr_op_time", "agr_debug_read", "agr_slab_ptr", "agr_synth_agent_id", "agr_synth_fill_host", "agr_synth_fill_rows", "agr_synth_bind_mint",
    "agr_agent_hash", "agr_agent_shard", "agr_comm_unique_id", "agr_comm_init", "agr_ingest_sharded", "agr_complete_sharded", "agr_snapshot", "agr_restore", "agr_verify", "agr_store_response_body", "agr_get_response_body",
    "agr_store_response", "agr_store_error_text", "agr_get_record_json", "agr_pending_json", "agr_rows_json", "agr_expire", "agr_reclaim", "agr_set_agent_states", "agr_json_decode",
    "agr_submit_ingest", "agr_submit_complete", "agr_poll", "agr_wait", "agr_ring_capacity", "agr_ingest_sharded_rows", "agr_fill_rows", "agr_reclaim_async",
    "agr_submit_ingest_var",
]

_lib = None


class AgrError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"agr error {code}: {msg}")
        self.code = code


def load_library(path: Optional[str] = None) -> C.CDLL:
    """Load libagentainer_b200.so (building it first if the sources are newer).  Fails loudly: no fallback."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or lib_path()
    if path is None:
        try:
            p = build_native()
        except RuntimeError:
            if not os.path.exists(p):
                raise
    lib = C.CDLL(p)
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
    sig = {
        "agr_create": (i32, [C.POINTER(AgrConfig), C.POINTER(vp)]),
        "agr_destroy": (None, [vp]),
        "agr_abi_version": (u32, []),
        "agr_last_error": (C.c_char_p, []),
        "agr_strerror": (C.c_char_p, [i32]),
        "agr_set_agent_state": (i32, [vp, C.c_char_p, C.c_uint8]),
        "agr_drop_agent": (i32, [vp, C.c_char_p]),
        "agr_agent_slot": (i32, [vp, C.c_char_p]),
        "agr_ingest": (i32, [vp, vp, u32, vp, C.POINTER(u64)]),
        "agr_ingest_ex": (i32, [vp, vp, u32, vp, vp, C.POINTER(u64)]),
        "agr_ingest_var": (i32, [vp, vp, vp, u32, vp, vp, C.POINTER(u64)]),
        "agr_replay_scan_var": (i32, [vp, vp, vp, u64, vp, u32, C.POINTER(u32), C.POINTER(u64)]),
        "agr_get_record_var": (i32, [vp, C.c_char_p, vp, vp, u32, C.POINTER(u32)]),
        "agr_complete": (i32, [vp, vp, u32, vp]),
        "agr_replay_scan": (i32, [vp, vp, vp, u32, C.POINTER(u32)]),
        "agr_pending": (i32, [vp, C.c_char_p, vp, u32, C.POINTER(u32)]),
        "agr_get_record": (i32, [vp, C.c_char_p, vp, vp]),
        "agr_list": (i32, [vp, C.c_char_p, i32, vp, u32, C.POINTER(u32)]),
        "agr_stats_get": (i32, [vp, C.POINTER(AgrStats)]),
        "agr_host_alloc": (vp, [C.c_size_t]),
        "agr_host_free": (None, [vp]),
        "agr_mint_ids": (i32, [vp, u64, u32, vp]),
        "agr_reserve_rows": (i32, [vp, u32, C.POINTER(u64)]),
        "agr_ingest_rows": (i32, [vp, u64, u32, vp]),
        "agr_ingest_rows_async": (i32, [vp, u64, u32]),
        "agr_sync": (i32, [vp]),
        "agr_stream": (vp, [vp]),
        "agr_slab_ptr": (vp, [vp, u64]),
        "agr_debug_read": (i32, [vp, i32, u64, u32, vp]),
        "agr_op_time": (i32, [vp, i32, C.POINTER(C.c_double)]),
        "agr_kernel_time": (i32, [vp, C.POINTER(C.c_double), C.POINTER(u64)]),
        "agr_synth_agent_id": (i32, [C.POINTER(AgrSynth), u32, C.c_char_p]),
        "agr_synth_fill_host": (i32, [C.POINTER(AgrSynth), u64, u32, vp]),
        "agr_synth_fill_rows": (i32, [vp, C.POINTER(AgrSynth), u64, u64, u32]),
        "agr_synth_bind_mint": (i32, [vp, C.POINTER(AgrSynth), u64]),
        "agr_agent_hash": (u64, [C.c_char_p]),
        "agr_agent_shard": (u32, [C.c_char_p, u32]),
        "agr_store_response_body": (i32, [vp, C.c_char_p, vp, vp, u32]),
        "agr_get_response_body": (i32, [vp, C.c_char_p, vp, vp, u32, C.POINTER(u32)]),
        "agr_store_response": (i32, [vp, C.c_char_p, vp, vp, u32, vp, u32]),
        "agr_store_error_text": (i32, [vp, C.c_char_p, vp, vp, u32]),
        "agr_get_record_json": (i32, [vp, C.c_char_p, vp, vp, u32, C.POINTER(u32)]),
        "agr_pending_json": (i32, [vp, C.c_char_p, vp, u64, C.POINTER(u64), C.POINTER(u32)]),
        "agr_rows_json": (i32, [vp, u64, u32, i32, vp, u64, C.POINTER(u64), vp]),
        "agr_snapshot": (i32, [vp, C.c_char_p]),
        "agr_restore": (i32, [C.POINTER(AgrConfig), C.c_char_p, C.POINTER(vp)]),
        "agr_verify": (i32, [vp, C.POINTER(u64), C.POINTER(u64)]),
        "agr_expire": (i32, [vp, u64, u64, C.POINTER(u64)]),
        "agr_reclaim": (i32, [vp, C.POINTER(u64)]),
        "agr_reclaim_async": (i32, [vp, C.POINTER(u64)]),
        "agr_set_agent_states": (i32, [vp, vp, vp, u32, vp]),
        "agr_json_decode": (i32, [vp, u32, vp, u32, vp, u32, vp, u32, vp]),
        "agr_comm_unique_id": (i32, [vp]),
        "agr_comm_init": (i32, [vp, vp, i32, i32]),
        "agr_ingest_sharded": (i32, [vp, vp, u32, vp, C.POINTER(AgrExchangeInfo)]),
        "agr_complete_sharded": (i32, [vp, vp, u32, vp, C.POINTER(AgrExchangeInfo)]),
        "agr_ingest_sharded_rows": (i32, [vp, u64, u32, vp, C.POINTER(AgrExchangeInfo)]),
        "agr_fill_rows": (i32, [vp, u64, vp, u32]),
        "agr_submit_ingest_var": (i32, [vp, vp, u32, C.POINTER(u64)]),
        "agr_poll": (i32, [vp, u64, C.POINTER(AgrResult)]),
        "agr_wait": (i32, [vp, u64, C.POINTER(AgrResult)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    if lib.agr_abi_version() != 2:
        raise RuntimeError("ABI version mismatch")
    if path is None:
        _lib = lib
    return lib


def _check(lib, rc: int) -> int:
    if rc < 0:
        raise AgrError(rc, (lib.agr_last_error() or b"").decode())
    return rc


def _ptr(a: np.ndarray) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data)


def _synth(seed, n_agents, zipf_milli=0, dup_permille=0, agent_nanos0=0, mint=None) -> AgrSynth:
    s = AgrSynth(seed, n_agents, zipf_milli, dup_permille, 0, agent_nanos0, 0, 0, 0, 0)
    if mint is not None:          # (engine, base_rid): duplicates name engine-minted ids
        eng, base = mint
        _check(eng.lib, eng.lib.agr_synth_bind_mint(eng.h, C.byref(s), base))
    return s


def synth_fill_host(first_index: int, n: int, *, seed=1, n_agents=16, zipf_milli=0, dup_permille=0,
                    agent_nanos0=0, mint=None, out: Optional[np.ndarray] = None) -> np.ndarray:
    lib = load_library()
    if out is None:
        out = np.zeros(n, dtype=record_dtype)
    s = _synth(seed, n_agents, zipf_milli, dup_permille, agent_nanos0, mint)
    _check(lib, lib.agr_synth_fill_host(C.byref(s), first_index, n, _ptr(out)))
    return out


def synth_agent_id(k: int, *, agent_nanos0=0) -> str:
    lib = load_library()
    buf = C.create_string_buffer(32)
    s = _synth(0, 1, 0, 0, agent_nanos0)
    _check(lib, lib.agr_synth_agent_id(C.byref(s), k, buf))
    return buf.value.decode()


def json_decode(js: bytes):
    """agr_json_decode: the wire form back into (header fields, path, flattened headers, body, AgrDecoded, response headers,
    response body, error text).  Host only: needs no GPU."""
    lib = load_library()
    src = np.frombuffer(js, dtype=np.uint8).copy() if js else np.zeros(1, dtype=np.uint8)
    rec = np.zeros(8192, dtype=np.uint8)
    resp = np.zeros(1 << 16, dtype=np.uint8)
    err = np.zeros(1 << 12, dtype=np.uint8)
    d = AgrDecoded()
    rc = lib.agr_json_decode(_ptr(src), len(js), _ptr(rec), rec.size, _ptr(resp), resp.size, _ptr(err), err.size, C.byref(d))
    if rc < 0:
        return rc, None
    head = rec[:96].view(header_dtype)[0]
    pl, hl, bl = int(head["path_len"]), int(head["hdr_len"]), int(head["body_len"])
    pay = rec[96: 96 + pl + hl + bl].tobytes()
    return 0, dict(header=head, path=pay[:pl], headers=pay[pl:pl + hl], body=pay[pl + hl:], info=d,
                   resp_headers=resp[: d.resp_hdr_len].tobytes(), resp_body=resp[d.resp_hdr_len: d.resp_hdr_len + d.resp_body_len].tobytes(),
                   error=err[: d.error_len].tobytes(), record=rec[: d.record_len].copy())


def comm_unique_id() -> bytes:
    lib = load_library()
    buf = (C.c_uint8 * 128)()
    _check(lib, lib.agr_comm_unique_id(C.cast(buf, C.c_void_p)))
    return bytes(buf)


def agent_hash(agent_id: str) -> int:
    return load_library().agr_agent_hash(agent_id.encode())


def agent_shard(agent_id: str, n: int) -> int:
    return load_library().agr_agent_shard(agent_id.encode(), n)


class PinnedArray:
    """numpy view over agr_host_alloc memory (the zero-copy producer path)."""

    def __init__(self, lib, n: int, dtype):
        self.lib = lib
        nbytes = max(1, n * np.dtype(dtype).itemsize)
        self.ptr = lib.agr_host_alloc(nbytes)
        if not self.ptr:
            raise AgrError(K.AGR_ENOMEM, "agr_host_alloc failed")
        buf = (C.c_uint8 * nbytes).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=n)

    def free(self):
        if self.ptr:
            self.array = None
            self.lib.agr_host_free(self.ptr)
            self.ptr = None


class Engine:
    """One shard (one GPU) of the request engine.  Thin wrapper: every method is one C-ABI call."""

    def __init__(self, *, device=-1, slab_rows=1 << 16, max_agents=1024, max_batch=0, flags=0, table_slots=0,
                 log_entries=0, k1_variant=0, id_secret=0, vslab_bytes=0, resp_bytes=0, restore_from=None):
        self.lib = load_library()
        cfg = AgrConfig(device, flags, slab_rows, table_slots, max_agents, max_batch or min(slab_rows, 1 << 20),
                        log_entries, id_secret, vslab_bytes, resp_bytes, k1_variant, 0)
        self.mint = bool(flags & K.AGR_CFG_MINT_IDS)
        self.varlen = bool(flags & K.AGR_CFG_VARLEN)
        h = C.c_void_p()
        if restore_from is not None:
            _check(self.lib, self.lib.agr_restore(C.byref(cfg), restore_from.encode(), C.byref(h)))
        else:
            _check(self.lib, self.lib.agr_create(C.byref(cfg), C.byref(h)))
        self.h = h
        self.max_batch = cfg.max_batch

    def close(self):
        if self.h:
            self.lib.agr_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- agent table
    def set_agent_state(self, agent_id: str, status) -> int:
        code = K.AGENT_STATUS_CODES[status] if isinstance(status, str) else int(status)
        return _check(self.lib, self.lib.agr_set_agent_state(self.h, agent_id.encode(), code))

    def set_agent_states(self, agent_ids, statuses) -> np.ndarray:
        """Bulk status feed (state sync): returns the slot (or negative error) per agent."""
        n = len(agent_ids)
        ids = np.zeros((n, 32), dtype=np.uint8)
        for i, a in enumerate(agent_ids):
            b = a.encode()
            ids[i, : len(b)] = np.frombuffer(b, dtype=np.uint8)
        st = np.array([K.AGENT_STATUS_CODES[s] if isinstance(s, str) else int(s) for s in statuses], dtype=np.uint8)
        slots = np.zeros(n, dtype=np.int32)
        _check(self.lib, self.lib.agr_set_agent_states(self.h, _ptr(ids), _ptr(st), n, _ptr(slots)))
        return slots

    def drop_agent(self, agent_id: str) -> None:
        _check(self.lib, self.lib.agr_drop_agent(self.h, agent_id.encode()))

    def agent_slot(self, agent_id: str) -> int:
        return _check(self.lib, self.lib.agr_agent_slot(self.h, agent_id.encode()))

    # ---- K1
    def ingest_ex(self, recs: np.ndarray, out: np.ndarray, ids: np.ndarray) -> int:
        """agr_ingest_ex: verdicts and Request.IDs into caller arrays (pinned or not); returns first_rid."""
        assert recs.dtype == record_dtype and out.dtype == verdict_dtype and ids.dtype == np.uint8 and ids.shape[1] == 16
        first = C.c_uint64()
        _check(self.lib, self.lib.agr_ingest_ex(self.h, _ptr(recs), len(recs), _ptr(out), _ptr(ids), C.byref(first)))
        return first.value

    def ingest(self, recs: np.ndarray, want_verdicts: bool = True, out: Optional[np.ndarray] = None) -> Tuple[Optional[np.ndarray], int]:
        assert recs.dtype == record_dtype and recs.flags["C_CONTIGUOUS"]
        n = len(recs)
        if out is not None:
            assert out.dtype == verdict_dtype and len(out) >= n
            want_verdicts = True
        else:
            out = np.zeros(n, dtype=verdict_dtype) if want_verdicts else None
        first = C.c_uint64()
        _check(self.lib, self.lib.agr_ingest(self.h, _ptr(recs), n, _ptr(out) if want_verdicts else None, C.byref(first)))
        return out, first.value

    def mint_ids(self, first_rid: int, n: int) -> np.ndarray:
        ids = np.zeros((n, 16), dtype=np.uint8)
        _check(self.lib, self.lib.agr_mint_ids(self.h, first_rid, n, _ptr(ids)))
        return ids

    def reserve_rows(self, n: int) -> int:
        first = C.c_uint64()
        _check(self.lib, self.lib.agr_reserve_rows(self.h, n, C.byref(first)))
        return first.value

    def ingest_rows(self, first_rid: int, n: int, want_verdicts: bool = True) -> Optional[np.ndarray]:
        out = np.zeros(n, dtype=verdict_dtype) if want_verdicts else None
        _check(self.lib, self.lib.agr_ingest_rows(self.h, first_rid, n, _ptr(out) if want_verdicts else None))
        return out

    def ingest_rows_async(self, first_rid: int, n: int) -> None:
        _check(self.lib, self.lib.agr_ingest_rows_async(self.h, first_rid, n))

    def sync(self) -> None:
        _check(self.lib, self.lib.agr_sync(self.h))

    def stream(self) -> int:
        return self.lib.agr_stream(self.h) or 0

    def kernel_time(self) -> Tuple[float, int]:
        ms, n = C.c_double(), C.c_uint64()
        _check(self.lib, self.lib.agr_kernel_time(self.h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def op_time(self, which: int) -> float:
        ms = C.c_double()
        _check(self.lib, self.lib.agr_op_time(self.h, which, C.byref(ms)))
        return ms.value

    def debug_read(self, which: str, first_rid: int, n: int) -> np.ndarray:
        sel = {"state": 0, "route": 1, "aux": 2, "cksum": 3}[which]
        out = np.zeros(n, dtype=np.uint64 if sel == 3 else np.uint32)
        _check(self.lib, self.lib.agr_debug_read(self.h, sel, first_rid, n, _ptr(out)))
        return out

    def slab_ptr(self, rid: int) -> int:
        return self.lib.agr_slab_ptr(self.h, rid) or 0

    def synth_fill_rows(self, first_index: int, first_rid: int, n: int, *, seed=1, n_agents=16, zipf_milli=0,
                        dup_permille=0, agent_nanos0=0, mint_base=None) -> None:
        s = _synth(seed, n_agents, zipf_milli, dup_permille, agent_nanos0, (self, mint_base) if mint_base is not None else None)
        _check(self.lib, self.lib.agr_synth_fill_rows(self.h, C.byref(s), first_index, first_rid, n))

    def pinned(self, n: int, dtype=record_dtype) -> PinnedArray:
        return PinnedArray(self.lib, n, dtype)

    # ---- variable-length records (AGR_CFG_VARLEN)
    def ingest_var(self, blob: np.ndarray, offsets: np.ndarray):
        assert blob.dtype == np.uint8 and offsets.dtype == np.uint32
        n = len(offsets) - 1
        out = np.zeros(n, dtype=verdict_dtype)
        ids = np.zeros((n, 16), dtype=np.uint8)
        first = C.c_uint64()
        _check(self.lib, self.lib.agr_ingest_var(self.h, _ptr(blob), _ptr(offsets), n, _ptr(out), _ptr(ids), C.byref(first)))
        return out, ids, first.value

    def submit_ingest_var(self, rec: np.ndarray) -> Optional[int]:
        """agr_submit_ingest_var: ONE record in the agr_ingest_var wire form; the ticket, or None on AGR_EAGAIN (collect, then again)."""
        assert rec.dtype == np.uint8 and rec.flags["C_CONTIGUOUS"]
        t = C.c_uint64()
        rc = self.lib.agr_submit_ingest_var(self.h, _ptr(rec), len(rec), C.byref(t))
        if rc == K.AGR_EAGAIN:
            return None
        _check(self.lib, rc)
        return t.value

    def poll(self, ticket: int, wait: bool = False):
        """agr_poll (agr_wait with wait=True): (verdict, request id, row, result) of a record's ticket, or None while undecided."""
        r = AgrResult()
        rc = (self.lib.agr_wait if wait else self.lib.agr_poll)(self.h, ticket, C.byref(r))
        if rc == K.AGR_EAGAIN:
            return None
        _check(self.lib, rc)
        return np.frombuffer(bytes(r.verdict), dtype=verdict_dtype)[0], bytes(r.request_id), r.rid, r.result

    def replay_scan_var(self, cap: int = 1 << 14, blob_cap: int = 1 << 24):
        while True:
            disp = np.zeros(cap, dtype=dispatch_dtype)
            blob = np.zeros(blob_cap, dtype=np.uint8)
            offs = np.zeros(cap + 1, dtype=np.uint64)
            n, nb = C.c_uint32(), C.c_uint64()
            rc = self.lib.agr_replay_scan_var(self.h, _ptr(disp), _ptr(blob), blob_cap, _ptr(offs), cap, C.byref(n), C.byref(nb))
            if rc == K.AGR_ECAP:
                cap, blob_cap = max(cap, int(n.value)), max(blob_cap, int(nb.value) + 16)
                continue
            _check(self.lib, rc)
            return disp[: n.value], blob[: nb.value], offs[: n.value + 1]

    def get_record_var(self, agent_id: str, request_id: bytes) -> Optional[np.ndarray]:
        out = np.zeros(8192, dtype=np.uint8)
        rid = (C.c_uint8 * 16).from_buffer_copy(request_id)
        ln = C.c_uint32()
        rc = self.lib.agr_get_record_var(self.h, agent_id.encode(), C.cast(rid, C.c_void_p), _ptr(out), 8192, C.byref(ln))
        if rc == K.AGR_ENOTFOUND:
            return None
        _check(self.lib, rc)
        return out[: ln.value]

    # ---- K4 (multi-GPU exchange)
    def comm_init(self, unique_id: bytes, rank: int, world: int) -> None:
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        _check(self.lib, self.lib.agr_comm_init(self.h, C.cast(buf, C.c_void_p), rank, world))

    def ingest_sharded(self, recs: np.ndarray, want_verdicts: bool = True):
        assert recs.dtype == record_dtype and recs.flags["C_CONTIGUOUS"]
        n = len(recs)
        out = np.zeros(n, dtype=verdict_dtype) if want_verdicts else None
        info = AgrExchangeInfo()
        _check(self.lib, self.lib.agr_ingest_sharded(self.h, _ptr(recs) if n else None, n, _ptr(out) if (want_verdicts and n) else None, C.byref(info)))
        return out, info

    def fill_rows(self, first_rid: int, recs: np.ndarray) -> None:
        assert recs.dtype == record_dtype and recs.flags["C_CONTIGUOUS"]
        _check(self.lib, self.lib.agr_fill_rows(self.h, first_rid, _ptr(recs), len(recs)))

    def ingest_sharded_rows(self, first_rid: int, n: int, want_verdicts: bool = False):
        """agr_ingest_sharded over rows already resident on the device (agr_reserve_rows + a device-side fill)."""
        out = np.zeros(n, dtype=verdict_dtype) if want_verdicts else None
        info = AgrExchangeInfo()
        _check(self.lib, self.lib.agr_ingest_sharded_rows(self.h, first_rid, n, _ptr(out) if want_verdicts and n else None, C.byref(info)))
        return out, info

    def complete_sharded(self, outs: np.ndarray):
        assert outs.dtype == outcome_dtype and outs.flags["C_CONTIGUOUS"]
        n = len(outs)
        res = np.zeros(n, dtype=np.int32)
        info = AgrExchangeInfo()
        _check(self.lib, self.lib.agr_complete_sharded(self.h, _ptr(outs) if n else None, n, _ptr(res) if n else None, C.byref(info)))
        return res, info

    # ---- K2
    def complete(self, outs: np.ndarray, want_results: bool = True) -> Optional[np.ndarray]:
        assert outs.dtype == outcome_dtype and outs.flags["C_CONTIGUOUS"]
        n = len(outs)
        res = np.zeros(n, dtype=np.int32) if want_results else None
        _check(self.lib, self.lib.agr_complete(self.h, _ptr(outs), n, _ptr(res) if want_results else None))
        return res

    # ---- K3
    def replay_scan(self, with_records: bool = True, cap: int = 1 << 16):
        while True:
            disp = np.zeros(cap, dtype=dispatch_dtype)
            recs = np.zeros(cap, dtype=record_dtype) if with_records else None
            n = C.c_uint32()
            rc = self.lib.agr_replay_scan(self.h, _ptr(disp), _ptr(recs) if with_records else None, cap, C.byref(n))
            if rc == K.AGR_ECAP:
                cap = int(n.value)
                continue
            _check(self.lib, rc)
            return disp[: n.value], (recs[: n.value] if with_records else None)

    def pending(self, agent_id: str, cap: int = 1 << 12) -> np.ndarray:
        while True:
            out = np.zeros(cap, dtype=record_dtype)
            n = C.c_uint32()
            rc = self.lib.agr_pending(self.h, agent_id.encode(), _ptr(out), cap, C.byref(n))
            if rc == K.AGR_ECAP:
                cap = int(n.value)
                continue
            _check(self.lib, rc)
            return out[: n.value]

    def get_record(self, agent_id: str, request_id: bytes) -> Optional[np.ndarray]:
        out = np.zeros(1, dtype=record_dtype)
        rid = (C.c_uint8 * 16).from_buffer_copy(request_id)
        rc = self.lib.agr_get_record(self.h, agent_id.encode(), C.cast(rid, C.c_void_p), _ptr(out))
        if rc == K.AGR_ENOTFOUND:
            return None
        _check(self.lib, rc)
        return out[0]

    def list(self, agent_id: str, which: int, cap: int = 1 << 12) -> np.ndarray:
        while True:
            ids = np.zeros((cap, 16), dtype=np.uint8)
            n = C.c_uint32()
            rc = self.lib.agr_list(self.h, agent_id.encode(), which, _ptr(ids), cap, C.byref(n))
            if rc == K.AGR_ECAP:
                cap = int(n.value)
                continue
            _check(self.lib, rc)
            return ids[: n.value]

    def store_response_body(self, agent_id: str, request_id: bytes, body: bytes) -> bool:
        rid = (C.c_uint8 * 16).from_buffer_copy(request_id)
        buf = (C.c_uint8 * max(1, len(body))).from_buffer_copy(body or b"\0")
        rc = self.lib.agr_store_response_body(self.h, agent_id.encode(), C.cast(rid, C.c_void_p), C.cast(buf, C.c_void_p), len(body))
        if rc == K.AGR_ENOTFOUND:
            return False
        _check(self.lib, rc)
        return True

    def store_response(self, agent_id: str, request_id: bytes, headers: bytes, body: bytes) -> bool:
        """requests.Response of StoreResponse (requests.go:142-147): flattened first-value headers + body."""
        rid = (C.c_uint8 * 16).from_buffer_copy(request_id)
        hb = (C.c_uint8 * max(1, len(headers))).from_buffer_copy(headers or b"\0")
        bb = (C.c_uint8 * max(1, len(body))).from_buffer_copy(body or b"\0")
        rc = self.lib.agr_store_response(self.h, agent_id.encode(), C.cast(rid, C.c_void_p), C.cast(hb, C.c_void_p), len(headers),
                                         C.cast(bb, C.c_void_p), len(body))
        if rc == K.AGR_ENOTFOUND:
            return False
        _check(self.lib, rc)
        return True

    def store_error_text(self, agent_id: str, request_id: bytes, text: bytes) -> bool:
        """Request.Error = err.Error() (requests.go:244)."""
        rid = (C.c_uint8 * 16).from_buffer_copy(request_id)
        tb = (C.c_uint8 * max(1, len(text))).from_buffer_copy(text or b"\0")
        rc = self.lib.agr_store_error_text(self.h, agent_id.encode(), C.cast(rid, C.c_void_p), C.cast(tb, C.c_void_p), len(text))
        if rc == K.AGR_ENOTFOUND:
            return False
        _check(self.lib, rc)
        return True

    def get_record_json(self, agent_id: str, request_id: bytes) -> Optional[bytes]:
        """The value of agent:{a}:requests:{r}: json.Marshal(requests.Request) (requests.go:101,170,265)."""
        rid = (C.c_uint8 * 16).from_buffer_copy(request_id)
        cap = 1 << 16
        while True:
            out = (C.c_uint8 * cap)()
            ln = C.c_uint32()
            rc = self.lib.agr_get_record_json(self.h, agent_id.encode(), C.cast(rid, C.c_void_p), C.cast(out, C.c_void_p), cap, C.byref(ln))
            if rc == K.AGR_ENOTFOUND:
                return None
            if rc == K.AGR_ECAP:
                cap = int(ln.value)
                continue
            _check(self.lib, rc)
            return bytes(out[: ln.value])

    def pending_json(self, agent_id: str) -> Tuple[bytes, int]:
        """json.Marshal(GetPendingRequests(agent)) (requests.go:197-225, server.go:646-650) and the entry count."""
        ln, cnt = C.c_uint64(), C.c_uint32()
        _check(self.lib, self.lib.agr_pending_json(self.h, agent_id.encode(), None, 0, C.byref(ln), C.byref(cnt)))
        out = np.zeros(max(1, ln.value), dtype=np.uint8)
        _check(self.lib, self.lib.agr_pending_json(self.h, agent_id.encode(), _ptr(out), out.size, C.byref(ln), C.byref(cnt)))
        return out[: ln.value].tobytes(), int(cnt.value)

    def rows_json(self, first_rid: int, n: int, as_array: bool = False, fetch: bool = True, roundtrip: bool = False):
        """Rows [first_rid, +n) in wire form.  fetch=False leaves the bytes on the device and returns only the length.
        roundtrip: strings as they read after a json.Unmarshal (what GetPendingRequests hands on)."""
        as_array = int(as_array) | (2 if roundtrip else 0)
        ln = C.c_uint64()
        _check(self.lib, self.lib.agr_rows_json(self.h, first_rid, n, int(as_array), None, 0, C.byref(ln), None))
        if not fetch:
            return int(ln.value)
        out = np.zeros(max(1, ln.value), dtype=np.uint8)
        offs = np.zeros(n + 1, dtype=np.uint64)
        _check(self.lib, self.lib.agr_rows_json(self.h, first_rid, n, int(as_array), _ptr(out), out.size, C.byref(ln), _ptr(offs)))
        return out[: ln.value].tobytes(), offs

    def get_response_body(self, agent_id: str, request_id: bytes) -> Optional[bytes]:
        rid = (C.c_uint8 * 16).from_buffer_copy(request_id)
        out = (C.c_uint8 * 65536)()
        ln = C.c_uint32()
        rc = self.lib.agr_get_response_body(self.h, agent_id.encode(), C.cast(rid, C.c_void_p), C.cast(out, C.c_void_p), 65536, C.byref(ln))
        if rc == K.AGR_ENOTFOUND:
            return None
        _check(self.lib, rc)
        return bytes(out[: ln.value])

    def snapshot(self, path: str) -> None:
        _check(self.lib, self.lib.agr_snapshot(self.h, path.encode()))

    def expire(self, now: int, ttl: int, want_count: bool = True) -> Optional[int]:
        """Drop the records whose last SET is ttl or more before now (the reference's 24 h key TTL); returns how many
        (want_count=False: no count, and the call does not wait for the sweep)."""
        if not want_count:
            _check(self.lib, self.lib.agr_expire(self.h, now, ttl, None))
            return None
        n = C.c_uint64()
        _check(self.lib, self.lib.agr_expire(self.h, now, ttl, C.byref(n)))
        return int(n.value)

    def reclaim(self) -> int:
        """AGR_CFG_RING: release the rows at the tail that hold no record any more; returns how many."""
        n = C.c_uint64()
        _check(self.lib, self.lib.agr_reclaim(self.h, C.byref(n)))
        return int(n.value)

    def reclaim_async(self) -> int:
        """agr_reclaim_async: releases what the previous call's scan found, starts the next scan; returns rows released now."""
        n = C.c_uint64()
        _check(self.lib, self.lib.agr_reclaim_async(self.h, C.byref(n)))
        return int(n.value)

    def verify(self) -> Tuple[int, int]:
        rows, bad = C.c_uint64(), C.c_uint64()
        _check(self.lib, self.lib.agr_verify(self.h, C.byref(rows), C.byref(bad)))
        return rows.value, bad.value

    def stats(self) -> dict:
        s = AgrStats()
        _check(self.lib, self.lib.agr_stats_get(self.h, C.byref(s)))
        return {n: getattr(s, n) for n, _ in AgrStats._fields_}
