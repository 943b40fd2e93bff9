// agr_svc.h — the single-request front end (AGR_CFG_COMBINE): shared layout of the pinned op ring between the calling
// threads, the dispatcher thread (agr_engine.cu) and the service kernel (agr_svc.cu).
//
// The reference serves one goroutine per HTTP request (net/http accept loop -> proxyToAgentHandler, server.go:493-573), so
// the call pattern at the boundary is "many OS threads, ONE request per call": agr_ingest_ex(n = 1) then agr_complete(n = 1).
// A kernel launch per call would cap the engine near 10^5 requests/s.  Instead:
//   callers     claim ring slots with one fetch_add, write their record / outcome into PINNED, device-mapped host memory,
//               publish the slot, and spin (then yield) on the slot's result word;  a variable-length record (AGR_CFG_VARLEN)
//               takes a RUN of ceil(len / 512) consecutive slots: continuation slots (SVC_OP_CONT) are published first, the
//               head slot (SVC_OP_RECORD) last, and its stored length goes into the per-slot length word before that;
//   dispatcher  one thread per handle: takes the contiguous published prefix of the ring (<= SVC_MAX_OPS, <= 128 record slots,
//               a run whole or not at all), reserves slab rows (and, AGR_CFG_VARLEN, slab bytes) for its records under the handle
//               mutex and publishes a 256 B batch descriptor;
//   service kernel  ONE resident CTA polls the descriptor ring over PCIe, pulls the batch's payloads straight out of host
//               memory, runs the K1 decision chain (records) and the K2 state machine (outcomes) of agr_device.cuh on them,
//               and writes verdict / id / row / result back into host memory.  No launch, no cudaMemcpy and no stream
//               synchronisation on the per-request path.
// Event order: batch by batch; inside a batch the records in ring order, then the outcomes in ring order.  All operations of
// one batch were in flight at the same time (none had returned), so this is a linearisation of the concurrent calls.
// Every other entry point stops the kernel first (it runs on the handle's stream), so the rest of the engine never sees it.
#pragma once
#include <stdint.h>

#define SVC_SLOTS 16384u          // ring slots (power of two)
#define SVC_MAX_OPS 256u          // ring slots per batch (<= 128 of them record slots: what one shared-memory stage of the kernel holds)
#define SVC_MAX_CALL 32u          // records / outcomes per call that go through the ring
#define SVC_DESCS 64u             // descriptor ring entries
#define SVC_PAYLOAD 512u          // bytes per slot: an agr_record, or an agr_outcome in the first 64 B

// SVC_OP_CONT: slot 2 .. k of a variable-length record's run (its head slot is the SVC_OP_RECORD right before them)
enum { SVC_OP_SKIP = 0, SVC_OP_RECORD = 1, SVC_OP_OUTCOME = 2, SVC_OP_CONT = 3 };

// batch descriptor (256 B = 64 words), written by the dispatcher (host), polled by the kernel: sixteen lanes read 16 B each
// in ONE poll; the kernel accepts it when the batch number matches and the check word agrees with the other 62 words (a poll
// that raced the host's stores sees a mix of old and new words and fails the check), so no second PCIe round trip is needed
struct __attribute__((aligned(64))) svc_desc {
    uint32_t kinds[SVC_MAX_OPS / 16];     // words 0..15: 2 bits per op, SVC_OP_*
    uint64_t from;                        // absolute number of the batch's first ring slot
    uint32_t count;                       // ops in the batch
    uint32_t n_records;                   // SVC_OP_RECORD ops among them: rows first_p .. first_p + n_records
    uint64_t first_l;                     // logical (arrival) number of the first record's row
    uint32_t first_p;                     // its physical row
    uint32_t tail_phys;                   // live window of the slab after this batch's rows were reserved
    uint64_t tail, head_l;
    uint64_t idx_base;
    uint64_t vbase;                       // AGR_CFG_VARLEN: physical slab byte offset of the first record (the others follow it in
                                          // ring order, each at the sum of the stored lengths before it)
    uint64_t reserved[14];
    uint64_t check;                       // words 60..61: XOR of svc_mix_word over words 0..59 and 62..63
    uint64_t seq;                         // words 62..63: batch number; the kernel waits for desc[seq % SVC_DESCS].seq == seq
};

static_assert(sizeof(svc_desc) == 256, "svc_desc must be 256 B (sixteen 16 B lanes)");

// per-slot result: ONE 16-byte store from the kernel (a single PCIe write inside one cache line: the caller sees all of it or
// none of it, so no system-wide fence sits between "result" and "done"):
//   record   w0, w1 = agr_verdict (w0's low byte = AGR_V_*, never 0);  w2 | (w3 & 0xffff) << 32 = logical row
//            host-side failure (slab full / CUDA error, written by the dispatcher): w0 = 0, w1 = (uint32_t)error code
//   outcome  w0 = (uint32_t)result (0 / AGR_ENOTFOUND / error code)
//   w3 >> 16 = tag of the slot's lap (svc_tag): the caller spins on it, and sets SVC_COLLECTED in it once it has read the
//              answer — that line is in the collector's cache anyway, so freeing a slot costs no extra miss.
//   continuation slot of a run: only the tag; it is written BEFORE the head's answer (so the collector's SVC_COLLECTED, which
//              it sets in every cell of the run, can never be overwritten by it)
// Request.ID is not shipped: with engine-minted ids it is a function of the row (agr_mint_id, computed by the caller's
// thread), with caller-supplied ids the caller has it already.
struct __attribute__((aligned(16))) svc_res { volatile uint32_t w[4]; };
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline uint32_t svc_tag(uint64_t slot_abs) { return (uint32_t)((slot_abs / SVC_SLOTS) & 0x3fffu) + 1u; }   // 1 .. 16384
#define SVC_COLLECTED 0x8000u     // or-ed into the tag by whoever collected the answer: the slot may be written for the next lap

// control block (host memory): how the host stops the kernel and how the kernel says where it stopped
struct __attribute__((aligned(64))) svc_ctl {
    volatile uint32_t stop;               // host -> kernel: leave once no published batch is left
    volatile uint32_t state;              // kernel -> host: 1 running, 0 exited, 2 exited on the safety timeout
    volatile uint64_t done_seq;           // kernel -> host: last batch completed
    volatile uint64_t heartbeat;          // kernel -> host: polls so far (diagnostics)
    volatile uint64_t cyc_wait, cyc_load, cyc_work, cyc_publish;   // kernel -> host: SM cycles spent waiting for a batch, pulling
                                          // payloads, deciding, publishing results (diagnostics, AGR_SVC_DEBUG)
};

static_assert(sizeof(svc_res) == 16, "svc_res must be 16 B");

struct svc_dev {                          // device-visible addresses of the pinned ring (UVA: host pointer == device pointer)
    const svc_desc* desc;
    const uint8_t* payload;               // [SVC_SLOTS][SVC_PAYLOAD]
    const uint32_t* lens;                 // [SVC_SLOTS] AGR_CFG_VARLEN: stored length of the record whose run starts at the slot
    svc_res* res;                         // [SVC_SLOTS]
    svc_ctl* ctl;
    uint32_t* dupfix;                     // device word for in-batch duplicate ids (hash-id mode)
    unsigned long long idle_ns;           // safety: leave after this long without a batch even if nobody said stop
};
