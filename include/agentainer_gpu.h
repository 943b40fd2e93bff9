/*
 * agentainer_gpu.h — C-ABI of the B200-native request queue / replay / route engine.
 *
 * This is the drop-in boundary for ONE path of oso95/Agentainer-lab: the
 * internal/requests persistence + replay queue and the decision part of the
 * internal/api reverse proxy.  The reference has no FFI of its own (it is pure
 * Go talking to Redis); the seam is the Go method set of requests.Manager and
 * requests.ReplayWorker plus the decision code in proxyToAgentHandler.  Every
 * entry point below names the reference interface it replaces (file:line,
 * relative to the reference tree).  The cgo binding a maintainer adds is in
 * INTEGRATION.md.
 *
 * Conventions
 *   - plain C, no CUDA / torch types in any signature;
 *   - the caller owns every input buffer until the call returns; the library
 *     never retains a caller pointer (cgo pointer-passing rules);
 *   - outputs go to caller-allocated arrays with (cap, *n);
 *   - return 0 on success, a negative AGR_E* code otherwise; never aborts;
 *     agr_last_error() gives a thread-local message for the last failure;
 *   - every entry point is thread-safe (calls on one handle are linearised in
 *     the order they acquire the handle; that order IS the event order the
 *     state machine sees, like commands arriving at a single Redis server);
 *   - there is no CPU fallback: without a usable sm_100 device agr_create fails.
 */
#ifndef AGENTAINER_GPU_H
#define AGENTAINER_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AGR_ABI_VERSION 2u

/* ------------------------------------------------------------------ errors */
#define AGR_OK          0
#define AGR_EINVAL     -1   /* bad argument */
#define AGR_ENODEV     -2   /* no usable CUDA device (sm_100) */
#define AGR_ENOMEM     -3   /* host or device allocation failed */
#define AGR_ENOSPC     -4   /* slab / log / agent table capacity exhausted */
#define AGR_ENOTFOUND  -5   /* key miss: "failed to get request" (requests.go:153-156,232-235), unknown agent */
#define AGR_ECUDA      -6   /* CUDA runtime error (message in agr_last_error) */
#define AGR_ECAP       -7   /* caller's output array too small; *n holds the needed count */
#define AGR_ECOMM      -8   /* multi-GPU exchange (NCCL) error */
#define AGR_EAGAIN      1   /* not an error: agr_poll — the ticket has not been decided yet; agr_submit_* — the ring slot drawn still
                               holds an answer nobody has collected: agr_poll your outstanding tickets, then submit again */

/* ---------------------------------------------------------- record layout */
/*
 * Fixed-stride binary form of requests.Request (requests.go:27-41).  512 B,
 * little-endian, naturally aligned.  IDs and time are supplied by the caller:
 * the reference mints uuid.New() / time.Now() inside StoreRequest
 * (requests.go:87,96); the Go shim mints them before the call so that the
 * state machine is a pure function of its input stream.
 */
#define AGR_RECORD_BYTES   512u
#define AGR_HEADER_BYTES    96u
#define AGR_PAYLOAD_BYTES  (AGR_RECORD_BYTES - AGR_HEADER_BYTES)   /* 416 */
#define AGR_AGENT_ID_BYTES  32u   /* "agent-<unixnano>" (agent.go:594-596) NUL padded, <=31 chars */

/* flags */
#define AGR_F_REPLAY        0x00000001u  /* X-Agentainer-Replay: true (server.go:506) */
#define AGR_F_METHOD_SHIFT  8            /* bits 8..15: method code */
#define AGR_F_METHOD_MASK   0x0000ff00u
enum { AGR_M_GET = 1, AGR_M_POST = 2, AGR_M_PUT = 3, AGR_M_DELETE = 4, AGR_M_PATCH = 5, AGR_M_HEAD = 6, AGR_M_OPTIONS = 7 };

/* RequestStatus (requests.go:19-24) */
enum { AGR_ST_NONE = 0, AGR_ST_PENDING = 1, AGR_ST_PROCESSING = 2, AGR_ST_COMPLETED = 3, AGR_ST_FAILED = 4 };

typedef struct agr_record {
    uint8_t  request_id[16];   /* raw UUID bytes of Request.ID (fresh records: minted by the caller, must be unique and non-zero) */
    uint8_t  replay_of[16];    /* X-Agentainer-Request-ID of a replay-flagged request (server.go:519-522); all-zero = header absent */
    char     agent_id[AGR_AGENT_ID_BYTES];
    uint64_t seq;              /* logical created_at (requests.go:96): caller's arrival counter */
    uint32_t flags;            /* AGR_F_* */
    uint16_t path_len;         /* Request.Path, stored WITH the /agent/{id} prefix (Q3) and without the query (Q4) */
    uint16_t hdr_len;          /* flattened first-value headers "Key: Value\n" sorted by key (Q5) */
    uint32_t body_len;
    uint8_t  status;           /* AGR_ST_*; on input ignored; on output (agr_pending / agr_get_record) the live value */
    uint8_t  retry_count;      /* same */
    uint8_t  max_retries;      /* requests.go:95: 3; 0 on input means 3 */
    uint8_t  error_code;       /* output only: AGR_OUT_* kind that last failed it (Request.Error is a string in the reference) */
    uint16_t resp_status;      /* output only: Response.StatusCode of the stored response, 0 if none */
    uint16_t reserved0;
    uint32_t reserved1;
    uint8_t  payload[AGR_PAYLOAD_BYTES];  /* path | headers | body, zero padded; path_len+hdr_len+body_len <= 416 */
} agr_record;

/* ------------------------------------------------------------------ config */
#define AGR_CFG_PERSISTENCE   0x1u  /* features.request_persistence (config.go:70); default on */
#define AGR_CFG_TIMING        0x4u  /* record CUDA-event pairs around the dominant K1 kernel (agr_kernel_time) */
#define AGR_CFG_MINT_IDS      0x8u  /* the engine mints Request.ID itself, like StoreRequest does (requests.go:87): the id is an
                                       exact invertible function of the record's row, agr_record.request_id of fresh records is
                                       ignored on input, callers read the ids with agr_mint_ids.  No dedupe-index table exists in
                                       this mode (lookups decode the row and verify all 128 bits). */
#define AGR_CFG_COMBINE       0x20u /* single-request front end (SURVEY 8b threading: one goroutine per HTTP request, server.go:493): calls of
                                       agr_ingest / agr_ingest_ex / agr_complete with n <= 32 go through a lock-free ring in pinned,
                                       device-mapped host memory (one fetch_add per call), a dispatcher thread batches whatever is
                                       published, and ONE resident service kernel decides the batch and writes verdicts / ids / result
                                       codes straight back into host memory — no launch, copy or stream sync per request.  Event
                                       order: batch by batch; inside a batch records in ring order, then outcomes in ring order (all
                                       of them were in flight together).  With AGR_CFG_VARLEN the same holds for agr_ingest_var and
                                       agr_complete with n <= 32 (a record of stored length L takes ceil(L / 512) consecutive ring
                                       slots) and agr_submit_ingest_var; results are those of the batch calls. */
#define AGR_CFG_RING          0x40u /* the slab is a ring (with AGR_CFG_VARLEN the byte slab is a ring too): row ids keep counting arrivals, a
                                       record lives at row id mod slab_rows, and agr_reclaim hands the rows at the tail that no longer hold
                                       a record (agr_expire) back for reuse — a shard then runs indefinitely instead of filling up.
                                       A batch never wraps: rows left before the end of the slab are skipped (<= max_batch per lap;
                                       max_batch is clamped to slab_rows / 2).  With caller-supplied ids every agr_reclaim rebuilds the dedupe
                                       index from the live rows.  Without the flag the slab is append-only. */
#define AGR_CFG_VARLEN        0x10u /* variable-length records (BASELINE config 5): byte-addressed slab, agr_ingest_var / *_var reads */
#define AGR_CFG_DIAG_NO_INDEX  0x100u /* DIAGNOSTIC ONLY (results invalid): K1 skips the dedupe-index insert, to attribute kernel time */
#define AGR_CFG_DIAG_NO_CKSUM  0x200u /* DIAGNOSTIC ONLY (results invalid): K1 skips the record checksum */
#define AGR_CFG_SKIP_INFLIGHT 0x2u  /* EXTENSION, off in parity mode: replay scan skips records whose forward is still in flight (fixes Q16) */

typedef struct agr_config {
    int32_t  device;         /* CUDA ordinal; -1 = current */
    uint32_t flags;          /* AGR_CFG_*; 0 = AGR_CFG_PERSISTENCE */
    uint64_t slab_rows;      /* record capacity (rows of 512 B); 0 = 1<<20 */
    uint64_t table_slots;    /* dedupe-index slots, power of two >= 2*slab_rows; 0 = auto */
    uint32_t max_agents;     /* agent-table capacity; 0 = 4096 */
    uint32_t max_batch;      /* largest n accepted by one agr_ingest / agr_complete; 0 = 1<<20 */
    uint64_t log_entries;    /* capacity of the completed and failed logs; 0 = 2*slab_rows */
    uint64_t id_secret;      /* AGR_CFG_MINT_IDS: key of the id permutation; 0 = drawn from the OS CSPRNG at agr_create */
    uint64_t vslab_bytes;    /* AGR_CFG_VARLEN: capacity of the byte slab; 0 = 1024 * slab_rows */
    uint64_t resp_bytes;     /* capacity of the stored-response byte slab; 0 = 64 * slab_rows */
    uint32_t k1_variant;     /* 0 = default K1 kernel (TMA, 14 warps x 1 stage, fused index); 1..4 TMA shapes, 5 = LSU kernel,
                                | 0x10 = split stream / index kernels, | 0x20 = LSU form of the variable-length kernel —
                                alternates kept for A/B measurement; bits 8..15 = L2 prefetch distance of the TMA kernel;
                                bits 16..23 = k: AGR_CFG_TIMING times every k-th K1 launch (0, 1 = every launch) */
    uint32_t reserved;
} agr_config;

typedef struct agr_handle agr_handle;

/* --------------------------------------------------------------- lifecycle */
/* replaces requests.NewManager (requests.go:57) + NewReplayWorker (replay_worker.go:24): ONE process-wide
 * handle instead of the two stateless Managers the reference creates (server.go:62, main.go:335). */
int  agr_create(const agr_config* cfg, agr_handle** out);
void agr_destroy(agr_handle* h);
uint32_t agr_abi_version(void);
const char* agr_last_error(void);
const char* agr_strerror(int code);

/* ------------------------------------------------------------- agent table */
/* Agent status mirror.  Replaces the per-request GET agent:{id} + Unmarshal of agent.Manager.GetAgent
 * (agent.go:372-390) read at server.go:498 and replay_worker.go:166-189.  Called from wherever the host
 * writes Agent.Status (saveAgent agent.go:510-530, state sync).  Registers the agent on first use; slots are
 * handed out in registration order.  Returns the slot (>= 0) or a negative error. */
enum { AGR_AGENT_CREATED = 0, AGR_AGENT_RUNNING = 1, AGR_AGENT_STOPPED = 2, AGR_AGENT_PAUSED = 3, AGR_AGENT_FAILED = 4 };  /* agent.go:23-29 */
int agr_set_agent_state(agr_handle* h, const char* agent_id, uint8_t status);
/* The same for a batch of status writes (the periodic state sync, sync/state_sync.go:190-210, and quick sync,
 * pkg/agentsync/quick_sync.go:89-102, walk every agent): ids are fixed-stride NUL-padded strings; slots (nullable)
 * receives the slot or the negative error of each entry; the return value is 0 or the first error.  More than 16
 * entries are applied to the host mirror and uploaded as two table copies instead of one small copy per agent. */
int agr_set_agent_states(agr_handle* h, const char (*agent_ids)[AGR_AGENT_ID_BYTES], const uint8_t* statuses, uint32_t n, int32_t* slots);
/* replaces the queue cleanup of agent.Manager.Remove (agent.go:343-359): DEL agent:{id} and the three lists.
 * Records are left orphaned exactly like the reference (Q17). */
int agr_drop_agent(agr_handle* h, const char* agent_id);
int agr_agent_slot(agr_handle* h, const char* agent_id);   /* slot or AGR_ENOTFOUND */

/* ------------------------------------------------------- K1 ingest + route */
/* verdict codes = the HTTP decision of proxyToAgentHandler (server.go:493-557) */
enum {
    AGR_V_FORWARD     = 1,   /* agent running: reverse-proxy to http://{id}:8000 (server.go:546-572) */
    AGR_V_QUEUED      = 2,   /* 202, "Request queued for replay" (server.go:526-536) */
    AGR_V_UNAVAILABLE = 3,   /* 503 (server.go:539-540) */
    AGR_V_NOT_FOUND   = 4    /* 404 agent not found (server.go:499-502) */
};
#define AGR_VF_STORED   0x01u  /* StoreRequest ran: record persisted + RPUSH pending (requests.go:100-114) */
#define AGR_VF_TRACKED  0x02u  /* requestID != "" : completion will be recorded (server.go:588,597) */
#define AGR_VF_REPLAY   0x04u  /* replay-flagged: not stored again (server.go:508,519) */
#define AGR_VF_KNOWN    0x08u  /* replay-flagged and replay_of names a record stored earlier (dedupe hit) */
#define AGR_VF_DUP_ID   0x10u  /* fresh record whose request_id already exists: contract violation, handled as a
                                  persistence failure (server.go:511-514): not stored, untracked */
#define AGR_VF_BAD_LEN  0x20u  /* path_len + hdr_len + body_len exceeds the record's payload (416 B fixed form, stored length - 96
                                  variable-length form): the record cannot be persisted; handled like a StoreRequest error
                                  (server.go:511-514, Q20): not stored, untracked, the request itself still gets its verdict */

typedef struct agr_verdict {
    uint8_t  code;        /* AGR_V_* */
    uint8_t  flags;       /* AGR_VF_* */
    uint16_t http_status; /* 0 (forward), 202, 503, 404 */
    uint32_t agent_slot;  /* valid unless NOT_FOUND */
} agr_verdict;

/* Batch form of the per-request sequence
 *   GetAgent -> isReplay -> StoreRequest -> status gate            (server.go:498-541, requests.go:64-117)
 * applied to recs[0..n) in array order.  n == 1 is the single-request call.  first_rid (nullable) receives
 * the slab row of recs[0]; record i lives in row first_rid + i.  recs may be pageable or pinned host memory. */
int agr_ingest(agr_handle* h, const agr_record* recs, uint32_t n, agr_verdict* out, uint64_t* first_rid);
/* Same, and also returns Request.ID of every record as the engine knows it (nullable): with AGR_CFG_MINT_IDS the ids
 * the engine minted (what StoreRequest returns in storedReq.ID, server.go:515), otherwise the caller's own ids echoed. */
int agr_ingest_ex(agr_handle* h, const agr_record* recs, uint32_t n, agr_verdict* out, uint8_t (*ids)[16], uint64_t* first_rid);

/* ------------------------------------------------------- K2 complete / fail */
enum {
    AGR_OUT_RESPONSE  = 1,  /* a response came back (ANY status code, Q6): Manager.StoreResponse (requests.go:120-194),
                               reached from interceptTransport.RoundTrip (server.go:588-594), the worker
                               (replay_worker.go:158) and the manual replay handler (server.go:739) */
    AGR_OUT_DIAL_ERR  = 2,  /* "connection refused" | "no such host" | "dial tcp": stays pending (server.go:600-605) */
    AGR_OUT_ERROR     = 3   /* any other error: Manager.MarkRequestFailed (requests.go:228-275), reached from
                               server.go:606-611, replay_worker.go:109-112, server.go:728-733 */
};
typedef struct agr_outcome {
    uint8_t  request_id[16];
    char     agent_id[AGR_AGENT_ID_BYTES];
    uint8_t  kind;          /* AGR_OUT_* */
    uint8_t  reserved0;
    uint16_t http_status;   /* Response.StatusCode for AGR_OUT_RESPONSE */
    uint32_t reserved1;
    uint64_t seq;           /* logical processed_at / received_at (requests.go:146,164) */
} agr_outcome;              /* 64 B */

/* Applies outs[0..n) in array order.  results (nullable) receives per outcome 0 or AGR_ENOTFOUND (the
 * "failed to get request" error the callers only log, Q20).  An all-zero request_id is a no-op
 * (t.requestID == "", server.go:588,597). */
int agr_complete(agr_handle* h, const agr_outcome* outs, uint32_t n, int32_t* results);

/* ------------------------------------------------- single requests without a blocked thread (AGR_CFG_COMBINE) */
/* The reference handles every HTTP request on its own goroutine (server.go:493); goroutines are not OS threads, and a cgo call
 * that blocks until the verdict is back would pin one OS thread per in-flight request.  These calls are the same single-request
 * operations as agr_ingest_ex(n = 1) / agr_complete(n = 1), split into "hand it over" and "collect": the goroutine submits,
 * parks on a channel, and a few reaper goroutines collect (INTEGRATION.md).  Event order is the front end's: batch by batch.
 *   agr_submit_ingest / agr_submit_complete  copy ONE record / outcome into the pinned request ring and return a ticket at once
 *                                            (tickets live in a ring of agr_ring_capacity() slots; AGR_EAGAIN when the slot drawn
 *                                            still holds an uncollected answer of a lap ago: poll, then submit again.  A submit
 *                                            never waits for another thread's ticket, so callers cannot deadlock each other)
 *   agr_poll    AGR_OK: *out is filled and the ticket is spent;  AGR_EAGAIN: not decided yet (the ticket stays valid)
 *   agr_wait    the same, spinning until decided (what agr_ingest_ex / agr_complete do internally)
 * A ticket must be collected exactly once.  AGR_EINVAL on an engine created without AGR_CFG_COMBINE. */
typedef uint64_t agr_ticket;
typedef struct agr_result {
    agr_verdict verdict;       /* record: the proxy decision (zeroed for an outcome) */
    uint8_t  request_id[16];   /* record: Request.ID as the engine knows it */
    uint64_t rid;              /* record: its row */
    int32_t  result;           /* 0, AGR_ENOTFOUND (outcome: "failed to get request"), AGR_ENOSPC (record: slab full), AGR_ECUDA */
    uint32_t is_outcome;
} agr_result;                  /* 40 B */
int agr_submit_ingest(agr_handle* h, const agr_record* rec, agr_ticket* ticket);
int agr_submit_complete(agr_handle* h, const agr_outcome* outcome, agr_ticket* ticket);
/* AGR_CFG_VARLEN | AGR_CFG_COMBINE: agr_submit_ingest for ONE variable-length record in the agr_ingest_var wire form (96 B header,
 * payload zero padded to 16 B; len = its stored length, a multiple of 16 in [96, AGR_VAR_MAX_RECORD], else AGR_EINVAL).  It takes
 * ceil(len / 512) consecutive ring slots; AGR_EAGAIN when any of them still holds an uncollected answer.  agr_poll / agr_wait
 * collect the ticket as usual.  agr_submit_ingest_var on a fixed-stride engine, and agr_submit_ingest on a variable-length one,
 * return AGR_EINVAL. */
int agr_submit_ingest_var(agr_handle* h, const uint8_t* rec, uint32_t len, agr_ticket* ticket);
int agr_poll(agr_handle* h, agr_ticket ticket, agr_result* out);
int agr_wait(agr_handle* h, agr_ticket ticket, agr_result* out);
uint32_t agr_ring_capacity(void);

/* ------------------------------------------------------------ K3 replay scan */
typedef struct agr_dispatch {
    uint64_t rid;           /* slab row */
    uint32_t agent_slot;
    uint32_t reserved;
    uint8_t  request_id[16];
} agr_dispatch;             /* 32 B */

/* One tick of ReplayWorker.processAgents (replay_worker.go:58-87) up to, not including, the HTTP call:
 * agents with a non-empty pending list (KEYS agent:*:requests:pending) that are running (isAgentRunning,
 * :166-189), their pending lists in FIFO order (GetPendingRequests, requests.go:197-225), minus entries with
 * status == processing or retry_count >= max_retries (:101).  Output is grouped by agent in ascending slot
 * order (Redis leaves the KEYS order undefined, Q9), FIFO inside each agent.  The host performs
 * replayRequest (:120-163) for each entry and reports back through agr_ingest (replay-flagged) and
 * agr_complete.  If recs != NULL the stored records are gathered into recs[0..*n) in the same order. */
int agr_replay_scan(agr_handle* h, agr_dispatch* out, agr_record* recs, uint32_t cap, uint32_t* n);

/* Manager.GetPendingRequests (requests.go:197-225) for one agent: FIFO, live status / retry patched in. */
int agr_pending(agr_handle* h, const char* agent_id, agr_record* out, uint32_t cap, uint32_t* n);

/* storage.Get("agent:{a}:requests:{r}") as used by server.go:661-662,687-688 (Q22). */
int agr_get_record(agr_handle* h, const char* agent_id, const uint8_t request_id[16], agr_record* out);

/* LRANGE agent:{a}:requests:{pending|completed|failed} 0 -1 — the ID sequences parity is defined on
 * (completed keeps the Q7 duplicates). */
enum { AGR_LIST_PENDING = 0, AGR_LIST_COMPLETED = 1, AGR_LIST_FAILED = 2 };
int agr_list(agr_handle* h, const char* agent_id, int which, uint8_t (*ids)[16], uint32_t cap, uint32_t* n);

/* ------------------------------------------------ variable-length records (AGR_CFG_VARLEN) */
/* A variable-length record is the 96-byte header of agr_record (same fields, same offsets) followed by its payload
 * path | headers | body, zero padded to a multiple of 16 bytes; its stored length is 96 + round16(path_len + hdr_len +
 * body_len) <= AGR_VAR_MAX_RECORD.  A batch is one contiguous blob of such records plus offsets[0..n] (bytes from the
 * start of the blob, offsets[n] = blob length; every offset a multiple of 16).  Semantics are those of agr_ingest_ex. */
#define AGR_VAR_MAX_RECORD 8192u
int agr_ingest_var(agr_handle* h, const uint8_t* blob, const uint32_t* offsets, uint32_t n, agr_verdict* out,
                   uint8_t (*ids)[16], uint64_t* first_rid);
/* agr_replay_scan for variable-length records: dispatch entries as usual; if blob != NULL the stored records are packed
 * into blob (capacity blob_cap bytes) with offsets[0..*n] (live status / retry / response patched into the headers).
 * AGR_ECAP if either capacity is too small (*n and *blob_bytes hold what is needed). */
int agr_replay_scan_var(agr_handle* h, agr_dispatch* out, uint8_t* blob, uint64_t blob_cap, uint64_t* offsets, uint32_t cap,
                        uint32_t* n, uint64_t* blob_bytes);
/* storage.Get for a variable-length record: copies it into out (cap bytes), *len = stored length. */
int agr_get_record_var(agr_handle* h, const char* agent_id, const uint8_t request_id[16], uint8_t* out, uint32_t cap, uint32_t* len);

/* ------------------------------------------------- stored responses (requests.go:142-147,165) */
/* StoreResponse keeps the whole response in the record (status, first-value headers, body).  agr_complete carries the
 * status on the hot path; the bytes (flattened "Key: Value\n" headers + body, caller's framing) go here, off the hot
 * path, and come back for GET /agents/{id}/requests/{reqId} (server.go:655-679).  The latest store wins, like the
 * reference's SET.  AGR_ENOTFOUND if the record does not exist. */
int agr_store_response_body(agr_handle* h, const char* agent_id, const uint8_t request_id[16], const uint8_t* bytes, uint32_t len);
/* The same with the two parts of requests.Response told apart (requests.go:44-49): headers = the first-value header map
 * flattened as "Key: Value\n" lines sorted by key (the form agr_record.payload uses), body = the raw body.  This is
 * what the JSON wire form below reads; agr_store_response_body(bytes) == agr_store_response(no headers, bytes). */
int agr_store_response(agr_handle* h, const char* agent_id, const uint8_t request_id[16], const uint8_t* headers, uint32_t hdr_len,
                       const uint8_t* body, uint32_t body_len);
/* Request.Error = err.Error() (requests.go:244): the text MarkRequestFailed stored last.  agr_complete carries only the
 * fact of the failure; the Go shim hands the text over here (off the hot path).  Without it the wire form says
 * "transport error".
 * Both stores append to one byte slab of agr_config.resp_bytes.  With AGR_CFG_RING the slab is a ring as well:
 * agr_reclaim moves its tail to the oldest bytes a live row still refers to.  Without the ring it is append-only.  When it
 * is full the stores fail with AGR_ENOSPC and the records keep working without the extra bytes. */
int agr_store_error_text(agr_handle* h, const char* agent_id, const uint8_t request_id[16], const char* text, uint32_t len);
int agr_get_response_body(agr_handle* h, const char* agent_id, const uint8_t request_id[16], uint8_t* out, uint32_t cap, uint32_t* len);

/* ------------------------------------------------- JSON wire form (K5, SURVEY 8f-1) */
/* The reference stores and serves records as json.Marshal(requests.Request) (requests.go:27-49,101,170,265): the value
 * of the Redis key agent:{a}:requests:{r} read by GET /agents/{id}/requests/{reqId} and the replay handler
 * (server.go:661-669,687-695), and the "pending" array of GET /agents/{id}/requests (server.go:626-652).  K5 produces
 * exactly those bytes on the device from the binary rows: struct field order, encoding/json string escaping (HTML-safe,
 * invalid UTF-8 -> U+FFFD, U+2028/9 escaped), header maps in key order, []byte as padded std base64, times as RFC 3339
 * with nanoseconds in UTC (agr_record.seq / agr_outcome.seq are read as Unix nanoseconds), omitempty on processed_at /
 * response / error.
 *   agr_get_record_json : the stored value of one record;            AGR_ENOTFOUND like storage.Get's miss
 *   agr_pending_json    : json.Marshal(GetPendingRequests(agent)) — "[{...},{...}]", or "null" for an empty list (the Go
 *                         slice is nil then, requests.go:204); *count = entries.  GetPendingRequests json.Unmarshals every
 *                         record first (requests.go:215-221), so invalid UTF-8 appears here as a raw U+FFFD, while the stored
 *                         value (agr_get_record_json) of a never-updated record still spells it \ufffd
 *   agr_rows_json       : rows [first_rid, first_rid + n) as an array (as_array & 1) or back to back with
 *                         offsets[0..n] (nullable); as_array & 2: strings in their after-Unmarshal form, like
 *                         agr_pending_json; rows that hold no stored record encode as null.  out == NULL
 *                         leaves the bytes on the device and only reports *len (sizing call / resident bench).
 * AGR_ECAP if cap is too small (*len holds the size needed). */
int agr_get_record_json(agr_handle* h, const char* agent_id, const uint8_t request_id[16], uint8_t* out, uint32_t cap, uint32_t* len);
int agr_pending_json(agr_handle* h, const char* agent_id, uint8_t* out, uint64_t cap, uint64_t* len, uint32_t* count);
int agr_rows_json(agr_handle* h, uint64_t first_rid, uint32_t n, int as_array, uint8_t* out, uint64_t cap, uint64_t* len, uint64_t* offsets);

/* The other direction, on the host: json.Unmarshal of that form (requests.go:159,216,238; server.go:669,695) into the
 * variable-length record form (96-byte header of agr_record + path | flattened headers | body, 16-byte rounded) plus the
 * fields that live outside the record.  Pure host code, no handle, no CUDA call: for migrating an existing Redis keyspace
 * and for checking what K5 produced.  Accepts what encoding/json accepts for this shape (members in any order, unknown
 * members skipped, every string escape, null for absent maps / slices / pointers, RFC 3339 times with any offset).
 * resp receives the flattened response headers followed by the response body; error receives Request.Error (not
 * NUL-terminated).  AGR_EINVAL: malformed or not representable (record longer than AGR_VAR_MAX_RECORD, agent id longer
 * than 31 bytes); AGR_ECAP: a buffer is too small (out holds the sizes needed). */
typedef struct agr_decoded {
    uint8_t  status, retry_count, max_retries, has_response;   /* AGR_ST_*; Request.RetryCount / MaxRetries; Response != nil */
    uint16_t resp_status, reserved;
    uint32_t record_len;                                       /* bytes written to record */
    uint32_t resp_hdr_len, resp_body_len, error_len;           /* bytes written to resp (headers, then body) and to error */
    uint32_t reserved2;
    uint64_t created_at, processed_at, received_at;            /* Unix nanoseconds; 0 = absent */
} agr_decoded;
int agr_json_decode(const uint8_t* json, uint32_t len, uint8_t* record, uint32_t record_cap, uint8_t* resp, uint32_t resp_cap,
                    char* error, uint32_t error_cap, agr_decoded* out);

/* ------------------------------------------------- durability (SURVEY 8f-2) */
/* What Redis persistence gave the reference (records and queues survive a server restart, docker-compose.yml:11-12):
 * agr_snapshot writes the live state (slab rows, per-row state words, completed / failed logs, agent table) to a file;
 * agr_restore creates a new engine from it (cfg gives the capacities; id mode and record form must match the snapshot).
 * In hash-id mode the dedupe index is not stored: it is rebuilt on the device from the restored rows. */
int agr_snapshot(agr_handle* h, const char* path);
int agr_restore(const agr_config* cfg, const char* path, agr_handle** out);
/* The 24 h TTL of the record keys (SET ... EX 24h at requests.go:106,175,270; every SET restarts it, Q11).  Times are the
 * callers' own clock: agr_record.seq for StoreRequest's SET, agr_outcome.seq for the SETs of StoreResponse /
 * MarkRequestFailed.  agr_expire drops every record whose last SET lies ttl or more before `now` (same unit as seq):
 * GET misses from then on (agr_get_record / agr_complete: AGR_ENOTFOUND, "failed to get request"), GetPendingRequests and
 * the replay scan skip it (requests.go:210-213), and — like in the reference — its id stays in the pending / completed /
 * failed lists (agr_list).  *expired (nullable) = records dropped by this call; with expired == NULL the call only enqueues
 * the sweep and returns (stream-ordered before any later call on the handle).  The sweep keeps a lower bound of the last-SET
 * times per 4096-row chunk, so a periodic call reads only the chunks that can hold something due.  Rows are not reclaimed. */
int agr_expire(agr_handle* h, uint64_t now, uint64_t ttl, uint64_t* expired);
/* AGR_CFG_RING: releases the rows at the tail of the ring that hold no record any more — everything up to the first row
 * whose record is still stored — and drops their entries from the completed / failed lists (a deviation from the
 * reference, where the ids of expired records stay listed forever, Q10: the lists of a long-running shard stay bounded
 * instead).  Ids of released rows are never valid again (a minted id is checked against the live window).  *released
 * (nullable) = rows handed back.  Typical use: agr_expire(now, 24 h) then agr_reclaim, from the same ticker. */
int agr_reclaim(agr_handle* h, uint64_t* released);
/* The same without a host round trip in the caller's way: releases what the scan started by the PREVIOUS call found and starts the
 * next scan.  For a ticker that maintains the ring every step (agr_expire(now, ttl, NULL); agr_reclaim_async(h, NULL)): the
 * release lags one step, nothing waits for the GPU. */
int agr_reclaim_async(agr_handle* h, uint64_t* released);
/* Integrity sweep: recomputes the checksum of every stored record on the device and compares it with the one K1 took at
 * ingest.  *bad = number of rows that differ (0 on a healthy slab). */
int agr_verify(agr_handle* h, uint64_t* rows_checked, uint64_t* bad);

/* ------------------------------------------------------------------- stats */
typedef struct agr_stats {
    uint64_t rows_used, rows_cap;
    uint64_t ingested, stored, replay_flagged, dedupe_hits, forwarded, queued, unavailable, not_found, dup_ids;
    uint64_t completions, completion_misses, failures, dead_lettered, dial_errors;
    uint64_t replay_scans, replay_dispatched;
    uint64_t completed_log_len, failed_log_len;
    uint64_t k1_launches, k2_launches, k3_launches, k4_launches;   /* kernels of this library launched so far */
    uint64_t k5_launches;
    uint64_t rows_tail;     /* AGR_CFG_RING: first row id that has not been released (0 otherwise); rows_used - rows_tail <= rows_cap */
    uint64_t malformed;     /* records rejected with AGR_VF_BAD_LEN */
    uint64_t log_overflow;  /* agr_complete batches whose completed / failed pushes did not fit the log (they returned AGR_ENOSPC) */
    uint64_t svc_batches, svc_ops;   /* AGR_CFG_COMBINE: batches formed by the dispatcher / single-request operations served */
    uint32_t agents, device;
} agr_stats;
int agr_stats_get(agr_handle* h, agr_stats* out);

/* ----------------------------------------------- pinned-host / resident path */
/* internal/storage moves to pinned host + HBM slabs: the zero-copy producer path.  The Go side fills records
 * directly into pinned memory obtained here and passes that pointer to agr_ingest (DMA without a bounce). */
void* agr_host_alloc(size_t bytes);
void  agr_host_free(void* p);

/* AGR_CFG_MINT_IDS: the ids the engine minted for rows [first_rid, first_rid + n) (pure host computation).  Record i of
 * an agr_ingest batch lives in row first_rid + i. */
int agr_mint_ids(agr_handle* h, uint64_t first_rid, uint32_t n, uint8_t (*ids)[16]);

/* Split form of agr_ingest for callers that keep the batch resident on the device (bench "value" leg, and the
 * receive side of the multi-GPU exchange): reserve rows, fill them (agr_synth_fill_rows or a DMA of the caller's
 * own), then run K1 over them.  verdicts may be NULL (they stay on the device). */
int agr_reserve_rows(agr_handle* h, uint32_t n, uint64_t* first_rid);
int agr_fill_rows(agr_handle* h, uint64_t first_rid, const agr_record* recs, uint32_t n);   /* DMA host records into reserved rows (no K1) */
int agr_ingest_rows(agr_handle* h, uint64_t first_rid, uint32_t n, agr_verdict* out);
/* launch-only variants: enqueue on the handle's stream and return without synchronising */
int agr_ingest_rows_async(agr_handle* h, uint64_t first_rid, uint32_t n);
int agr_sync(agr_handle* h);
void* agr_stream(agr_handle* h);                 /* cudaStream_t the kernels run on (for CUDA-event timing) */
/* With AGR_CFG_TIMING: device time of the dominant K1 kernel (k1_ingest) summed over the launches since the last
 * call (at most the latest 1024), from CUDA events recorded on the launching stream.  Synchronises. */
int agr_kernel_time(agr_handle* h, double* sum_ms, uint64_t* launches);
/* With AGR_CFG_TIMING: device time (CUDA events on the launching stream) of the most recent kernel group:
 * which = 0 the K2 kernels of the last agr_complete, 1 the K3 select kernels of the last scan / pending / list,
 * 2 the K5 kernels of the last JSON encode (measure + scan + emit, including the host's read of the total between them). */
int agr_op_time(agr_handle* h, int which, double* ms);
void* agr_slab_ptr(agr_handle* h, uint64_t rid); /* device address of a slab row */

/* ------------------------------------------------------------ multi-GPU exchange (K4) */
/* One handle per GPU; shard owner of an agent = agr_agent_shard(id, world).  Fresh traffic is steered to the owner by
 * the host when it parses /agent/{id} (server.go:494-495) and needs no collective.  Records that reach a non-owner shard
 * (BASELINE config 4: replay-flagged requests re-injected through another shard's proxy) are routed here:
 * the batch is DMA'd straight into its slab rows; K4 bins it by owner there, copies only the records owned by a PEER into the
 * send buffer (their rows are marked empty) and ONE grouped ncclSend/ncclRecv all-to-all over NVLink ships every peer segment
 * into rows reserved at its owner; K1 runs over the own rows while the exchange is in flight and over the received rows after
 * it, and the verdicts travel back the same way and are restored to the caller's order.
 * NCCL is loaded at run time (libnccl.so.2); without it agr_comm_init fails with AGR_ECOMM.  Collective: every rank of
 * the communicator must call agr_ingest_sharded the same number of times (n may be 0). */
int agr_comm_unique_id(uint8_t out[128]);                                          /* rank 0; ship to the other ranks */
int agr_comm_init(agr_handle* h, const uint8_t id[128], int rank, int world);
typedef struct agr_exchange_info {
    uint32_t world, rank;
    uint32_t n_local, n_sent, n_received;      /* records of the batch owned here / shipped / received from peers */
    uint32_t sent_to[32], received_from[32];
    uint64_t first_rid;                        /* rows [first_rid, +n) hold the caller's batch in arrival order; the rows of records
                                                  that were shipped to their owner are empty */
    uint64_t recv_first_rid;                   /* rows [recv_first_rid, +n_received): the records received, grouped by source rank */
} agr_exchange_info;
int agr_ingest_sharded(agr_handle* h, const agr_record* recs, uint32_t n, agr_verdict* out, agr_exchange_info* info);
/* The same exchange over a batch that is already resident in rows [first_rid, +n) (agr_reserve_rows + a fill on the device). */
int agr_ingest_sharded_rows(agr_handle* h, uint64_t first_rid, uint32_t n, agr_verdict* out, agr_exchange_info* info);
/* The same route for outcomes (cross-shard replay reconciliation): an outcome reported at a shard that does not own the
 * agent (the worker of shard A replayed through shard B's proxy) is shipped to the owner, applied there by K2 in
 * (own host first, then peers by rank) order, and its result code comes back.  Collective like agr_ingest_sharded. */
int agr_complete_sharded(agr_handle* h, const agr_outcome* outs, uint32_t n, int32_t* results, agr_exchange_info* info);

/* Diagnostic read-back of the per-row SoA words (tests, snapshot tooling): which = 0 state (u32), 1 route (u32),
 * 2 aux (u32), 3 checksum (u64).  out must hold n elements of that width. */
enum { AGR_DBG_STATE = 0, AGR_DBG_ROUTE = 1, AGR_DBG_AUX = 2, AGR_DBG_CKSUM = 3 };
int agr_debug_read(agr_handle* h, int which, uint64_t first_rid, uint32_t n, void* out);

/* -------------------------------------------------- synthetic stream (bench) */
/* Counter-based generator of BASELINE.json's synthetic streams; integer-only, identical on host and device. */
typedef struct agr_synth {
    uint64_t seed;
    uint32_t n_agents;        /* 16 / 256 */
    uint32_t zipf_milli;      /* 0 = uniform; 1200 = Zipf s=1.2 by rank */
    uint32_t dup_permille;    /* replay-flagged duplicates per 1000 records (C3: 100) */
    uint32_t mint;            /* 1: duplicates name their target by the id the engine mints for it (set by agr_synth_bind_mint) */
    uint64_t agent_nanos0;    /* agent k has id "agent-<agent_nanos0 + k*1000003>" */
    uint64_t mint_base_rid;   /* row of stream index 0 */
    uint64_t mint_secret;
    uint32_t mint_shard, mint_gen;
} agr_synth;
/* For engines created with AGR_CFG_MINT_IDS: make the stream's duplicates refer to engine-minted ids, assuming stream
 * index j will be ingested into row base_rid + j. */
int agr_synth_bind_mint(agr_handle* h, agr_synth* s, uint64_t base_rid);
int agr_synth_agent_id(const agr_synth* s, uint32_t k, char out[AGR_AGENT_ID_BYTES]);
int agr_synth_fill_host(const agr_synth* s, uint64_t first_index, uint32_t n, agr_record* out);
int agr_synth_fill_rows(agr_handle* h, const agr_synth* s, uint64_t first_index, uint64_t first_rid, uint32_t n);

/* shard owner of an agent: FNV-1a 64 of the id bytes, mod n_shards (SURVEY 8e).  Go: hash/fnv New64a. */
uint64_t agr_agent_hash(const char* agent_id);
uint32_t agr_agent_shard(const char* agent_id, uint32_t n_shards);

#ifdef __cplusplus
}
#endif
#endif /* AGENTAINER_GPU_H */
