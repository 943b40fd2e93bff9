// agr_engine.cu — host side of the engine and the C-ABI of include/agentainer_gpu.h.
//
// One agr_handle == one GPU shard: HBM slab + SoA state + dedupe index + logs + agent-table mirror, one stream.
// Calls are linearised by the handle mutex; the order in which calls take it is the event order the state
// machine sees (the reference's serialisation point is the single-threaded Redis server).
// There is NO CPU fallback: every state transition happens in the kernels of agr_kernels.cu.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <sys/random.h>
#include <nccl.h>      // types only: every NCCL symbol is resolved with dlopen/dlsym at run time
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <thread>
#include <condition_variable>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/agentainer_gpu.h"
#include "agr_kernels.cuh"
#include "agr_svc.h"
#include <atomic>
#include <chrono>
#include <immintrin.h>
#include <sched.h>
#include <time.h>
#include <sys/prctl.h>
#include "agr_ring.hpp"

static_assert(sizeof(agr_record) == 512, "agr_record must be 512 B");
static_assert(sizeof(agr_outcome) == 64, "agr_outcome must be 64 B");
static_assert(sizeof(agr_dispatch) == 32, "agr_dispatch must be 32 B");
static_assert(sizeof(agr_verdict) == 8, "agr_verdict must be 8 B");
static_assert(sizeof(agr_slot) == 32, "agr_slot must be 32 B");
static_assert(sizeof(agr_agent_key) == 48, "agr_agent_key must be 48 B");
static_assert(sizeof(agr_dop) == 32, "agr_dop must be 32 B");
static_assert(sizeof(agr_k2op) == 16, "agr_k2op must be 16 B");

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }

#define CK(call)                                                                                     \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess)                                                                       \
            return fail(AGR_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_));              \
    } while (0)

struct agr_handle {
    std::mutex mu;
    agr_config cfg{};
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;        // H2D of chunk k+1 overlaps K1 of chunk k (agr_ingest pipeline)
    std::vector<cudaEvent_t> chunk_ev;
    cudaStream_t d2h_stream = nullptr;         // verdicts / ids of chunk k go back while chunk k+1 comes in (PCIe is full duplex)
    std::vector<cudaEvent_t> out_ev;
    agr_verdict* d_verdicts = nullptr;         // [max_batch], written by k1_post
    agr_verdict* h_verdicts = nullptr;         // pinned [max_batch]
    uint8_t* d_ids = nullptr;                  // [max_batch][16] Request.ID per record (agr_ingest_ex)
    uint8_t* h_ids = nullptr;                  // pinned
    agr_dev d{};
    uint64_t rows_used = 0;   // LOGICAL rows handed out so far (ring: includes the rows skipped at a wrap)
    uint64_t tail = 0;        // ring: first logical row that has not been released
    uint32_t* d_log_scratch = nullptr; uint32_t* d_lc_chunks = nullptr;   // ring: log compaction
    uint64_t released_total = 0;
    uint32_t* d_reclaim_scratch = nullptr;                        // k_first_live: {offset found, ticket}
    uint8_t* d_reclaim = nullptr; uint8_t* h_reclaim = nullptr;   // agr_reclaim's scan result (device scratch / pinned copy)
    cudaEvent_t reclaim_ev = nullptr; bool reclaim_pending = false; uint64_t reclaim_bound = 0;
    uint32_t* dupfix_base = nullptr; uint32_t batch_phase = 0;   // two sets of per-batch words, used alternately
    uint64_t scan_lo = 0;     // every row below has left its pending list for good
    uint64_t sweep_clean = 0; // append-only slab: rows below were ingested when agr_expire last ran (their chunks' time bounds are exact)
    // host agent map + mirror
    std::unordered_map<std::string, uint32_t> slot_of;
    std::vector<std::string> agent_names;
    std::vector<uint8_t> agent_status;
    std::vector<agr_agent_key> akeys_host;
    std::vector<uint32_t> akey_index;          // slot -> index of its entry in the open-addressing key table
    // staging
    uint8_t* bounce[2] = {nullptr, nullptr};   // pinned, for pageable caller buffers
    cudaEvent_t bounce_ev[2] = {nullptr, nullptr};
    size_t bounce_bytes = 0;
    agr_dop* h_ops = nullptr;                  // pinned [16] (single-key lookups)
    agr_outcome* h_outs = nullptr;             // pinned [max_batch]
    agr_outcome* d_outs = nullptr;             // [max_batch]
    int32_t* h_results = nullptr;              // pinned [max_batch]
    agr_k2_scratch k2{}; uint32_t k2_cap = 0;   // K2 scratch sized for k2_cap outcomes
    uint32_t* d_hrid = nullptr;                // rows found by the single-key resolve (k_resolve)
    uint32_t* h_k2flag = nullptr;              // pinned: k2_append's overflow flag of the last batch
    agr_dop* d_ops = nullptr;
    std::vector<std::pair<uint64_t, uint64_t>> resv;   // rows handed out by agr_reserve_rows and not ingested yet: [first, end)
    // K3
    uint32_t* d_matrix = nullptr; size_t matrix_entries = 0;
    uint32_t* d_cta_matrix = nullptr; size_t cta_matrix_entries = 0;
    uint32_t* d_selmask = nullptr; size_t selmask_words = 0;   // one selection bit per scanned item (k3_mark -> k3_place)
    uint32_t* d_gtotal = nullptr; uint32_t* d_goff = nullptr;
    uint32_t* d_out_rid = nullptr; uint32_t* d_out_slot = nullptr; uint32_t out_cap = 0;
    uint32_t* d_min_inq = nullptr;
    uint8_t* d_gather = nullptr; size_t gather_bytes = 0;
    uint8_t* h_gather = nullptr; size_t h_gather_bytes = 0;
    uint32_t* h_small = nullptr;               // pinned scratch (>= 64 words)
    unsigned long long* d_cdf = nullptr; uint32_t cdf_n = 0;
    // launch accounting
    uint64_t k1_launches = 0, k2_launches = 0, k3_launches = 0, k4_launches = 0;
    uint64_t replay_scans = 0, replay_dispatched = 0;
    std::vector<void*> dev_allocs, host_allocs;
    alignas(64) unsigned char tmap[128];       // CUtensorMap of the slab for the TMA K1 variants
    // stored responses: byte slab + per-row (offset, length), written off the hot path
    uint8_t* d_resp = nullptr; uint64_t resp_used = 0, resp_cap = 0;   // bytes appended so far (ring: logical, pads included) / capacity
    uint64_t resp_tail = 0;                    // ring: logical offset of the oldest byte a live row still refers to
    unsigned long long* d_resp_off = nullptr; uint32_t* d_resp_len = nullptr;
    uint32_t* d_resp_hlen = nullptr;           // leading bytes of the stored response that are its flattened headers
    unsigned long long* d_err_off = nullptr; uint32_t* d_err_len = nullptr;   // Request.Error text, same byte slab
    // K5 (JSON wire form) scratch
    uint32_t* d_jlen = nullptr; unsigned long long* d_joff = nullptr; unsigned long long* d_jchunk = nullptr; uint32_t j_cap = 0;
    uint8_t* d_json = nullptr; uint64_t json_cap = 0;
    uint64_t k5_launches = 0;
    uint64_t expired_total = 0;                // records dropped by agr_expire so far
    // single-request front end (AGR_CFG_COMBINE): pinned op ring + dispatcher thread + resident service kernel (agr_svc.h)
    struct svc_host* svc = nullptr;
    // variable-length mode
    uint64_t vused = 0, vcap = 0;               // bytes appended so far (ring: logical, pads included) / capacity
    uint64_t vtail = 0;                        // ring: logical offset of the first byte that has not been released
    uint32_t* d_voffsets = nullptr; uint32_t* d_tile_first = nullptr;   // per-batch offsets [max_batch+1], tile index
    uint32_t* h_voffsets = nullptr;
    uint32_t* d_lens = nullptr; unsigned long long* d_goffs = nullptr;  // gather scratch [out_cap]
    uint32_t lens_cap = 0;
    // multi-GPU exchange (K4)
    ncclComm_t comm = nullptr; int rank = 0, world = 1;
    uint8_t* d_stage = nullptr;                // incoming batch before binning [max_batch * 512]
    uint8_t* d_send = nullptr;                 // owner-major send buffer [max_batch * 512]
    uint8_t* d_owner = nullptr; uint32_t* d_perm = nullptr;
    uint32_t* d_k4matrix = nullptr; uint32_t k4_nwarps = 0;
    uint32_t* d_k4cnt = nullptr;               // [4][32]: gtotal, goff(33 → second row pair), recv counts
    agr_verdict* d_xverd = nullptr;            // verdicts of local + received rows [2 * max_batch]
    agr_verdict* d_vback = nullptr;            // verdicts returned by owners, owner-major [max_batch]
    agr_verdict* d_vout = nullptr;             // caller-order verdicts [max_batch]
    // AGR_CFG_TIMING: CUDA-event pairs around the dominant K1 kernel, on the launching stream
    std::vector<cudaEvent_t> tev; uint64_t tev_next = 0, tev_read = 0, timing_calls = 0;
    cudaEvent_t op_ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // [0,1] last K2 group, [2,3] last K3 select group, [4,5] last K5 encode
    bool op_timed[3] = {false, false, false};
};
#define AGR_TIMING_RING 1024

template <typename T>
static int dev_alloc(agr_handle* h, T** p, size_t count, bool zero) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, count * sizeof(T));
    if (e != cudaSuccess) return fail(AGR_ENOMEM, std::string("cudaMalloc ") + std::to_string(count * sizeof(T)) + " B: " + cudaGetErrorString(e));
    if (zero) { e = cudaMemsetAsync(q, 0, count * sizeof(T), h->stream); if (e != cudaSuccess) return fail(AGR_ECUDA, cudaGetErrorString(e)); }
    h->dev_allocs.push_back(q);
    *p = (T*)q;
    return 0;
}
// grow-only scratch: replaces *p by a larger buffer and releases the old one (every user of the old buffer has been
// synchronised by then: the callers hold the handle mutex and the previous operation ended with a stream sync)
template <typename T>
static int dev_regrow(agr_handle* h, T** p, size_t count, bool zero) {
    T* old = *p;
    int rc = dev_alloc(h, p, count, zero);
    if (rc < 0) return rc;
    if (old) {
        cudaStreamSynchronize(h->stream);
        auto it = std::find(h->dev_allocs.begin(), h->dev_allocs.end(), (void*)old);
        if (it != h->dev_allocs.end()) h->dev_allocs.erase(it);
        cudaFree(old);
    }
    return 0;
}
template <typename T>
static int host_regrow(agr_handle* h, T** p, size_t count);
template <typename T>
static int host_alloc(agr_handle* h, T** p, size_t count) {
    void* q = nullptr;
    cudaError_t e = cudaHostAlloc(&q, count * sizeof(T), cudaHostAllocDefault);
    if (e != cudaSuccess) return fail(AGR_ENOMEM, std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
    h->host_allocs.push_back(q);
    *p = (T*)q;
    return 0;
}
template <typename T>
static int host_regrow(agr_handle* h, T** p, size_t count) {
    T* old = *p;
    int rc = host_alloc(h, p, count);
    if (rc < 0) return rc;
    if (old) {
        cudaStreamSynchronize(h->stream);
        auto it = std::find(h->host_allocs.begin(), h->host_allocs.end(), (void*)old);
        if (it != h->host_allocs.end()) h->host_allocs.erase(it);
        cudaFreeHost(old);
    }
    return 0;
}
#define TRY(x) do { int r_ = (x); if (r_ < 0) return r_; } while (0)

// K2 scratch for up to n outcomes per batch
static int k2_scratch_alloc(agr_handle* h, size_t n) {
    TRY(dev_alloc(h, &h->k2.ops, n, false));
    TRY(dev_alloc(h, &h->k2.nxt, n, false));
    TRY(dev_alloc(h, &h->k2.eff, n + 8, false));
    TRY(dev_alloc(h, &h->k2.results, n, false));
    // word 0 = {ticket, overflow}, then one look-back word per tile: agr_launch_k2 clears the prefix a batch uses
    unsigned long long* words = nullptr;
    TRY(dev_alloc(h, &words, (size_t)agr_k2_tiles((uint32_t)n) + 2, true));
    h->k2.ticket = (uint32_t*)words;
    h->k2.overflow = h->k2.ticket + 1;
    h->k2.tiles = words + 1;
    h->k2_cap = (uint32_t)n;
    return 0;
}

// ---- logical rows (arrival numbers, what the API speaks) vs physical rows (where the record lives; see agr_dev)
static inline bool is_ring(const agr_handle* h) { return (h->cfg.flags & AGR_CFG_RING) != 0; }
static inline uint64_t phys_row(const agr_handle* h, uint64_t l) { return is_ring(h) ? l % h->cfg.slab_rows : l; }
static inline uint64_t rows_span(const agr_handle* h) {       // physical rows that have ever been handed out
    return is_ring(h) ? std::min<uint64_t>(h->rows_used, h->cfg.slab_rows) : h->rows_used;
}
static inline void sync_window(agr_handle* h) {               // the live window the kernels check decoded ids against
    h->d.tail = h->tail; h->d.head_l = h->rows_used;
    h->d.ring_rows = is_ring(h) ? (uint32_t)h->cfg.slab_rows : 0u;
    h->d.tail_phys = is_ring(h) ? (uint32_t)(h->tail % h->cfg.slab_rows) : 0u;
}

struct nccl_api {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static nccl_api g_nccl;
// pageable -> pinned staging copy.  One core moves ~13 GB/s, a quarter of what the link takes; big pieces are split over a
// few short-lived threads (the pinned path, agr_host_alloc, needs none of this).
static void par_memcpy(void* dst, const void* src, size_t bytes) {
    const size_t min_slice = (size_t)4 << 20;
    unsigned nt = (unsigned)std::min<size_t>(4, bytes / min_slice);
    if (nt <= 1) { memcpy(dst, src, bytes); return; }
    const size_t slice = ((bytes / nt) + 63) & ~(size_t)63;
    std::vector<std::thread> th;
    for (unsigned t = 1; t < nt; ++t) {
        const size_t o = (size_t)t * slice;
        if (o >= bytes) break;
        th.emplace_back([=] { memcpy((uint8_t*)dst + o, (const uint8_t*)src + o, std::min(slice, bytes - o)); });
    }
    memcpy(dst, src, std::min(slice, bytes));
    for (auto& x : th) x.join();
}
static bool is_pinned(const void* p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) == cudaSuccess) return attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    return false;
}

static uint64_t next_pow2(uint64_t v) { uint64_t p = 1; while (p < v) p <<= 1; return p; }

static void pack_agent_id(const char* id, unsigned long long w[4]) {
    char buf[AGR_AGENT_ID_BYTES];
    memset(buf, 0, sizeof buf);
    strncpy(buf, id, AGR_AGENT_ID_BYTES - 1);
    memcpy(w, buf, 32);
}


// ------------------------------------------------------------------------------------------ single-request front end
// Host side of agr_svc.h.  Lock-free for the callers: one fetch_add claims ring slots, the payload is written into pinned
// device-mapped memory, a release store publishes it, and the caller waits on a word the GPU writes.  One dispatcher thread
// per handle turns the published prefix of the ring into batch descriptors; the resident service kernel (k_svc) does the rest.
extern "C" { static int reserve_rows_locked(agr_handle* h, uint32_t n, uint64_t* first);
             static int reserve_var_locked(agr_handle* h, uint32_t n, uint64_t bytes, uint64_t* first, uint64_t* base); }
cudaError_t agr_launch_svc(const agr_dev& d, const svc_dev& v, const agr_k2_scratch& k2, unsigned long long next_seq, bool var, cudaStream_t st);
unsigned long long agr_svc_desc_check(const svc_desc* dsc);

struct svc_host {
    // ---- read-mostly (every caller reads these on every call; nothing here is written while callers run)
    svc_desc* desc = nullptr; uint8_t* payload = nullptr; svc_res* res = nullptr; svc_ctl* ctl = nullptr;   // pinned, device-mapped
    std::atomic<uint32_t>* ready = nullptr;             // [SVC_SLOTS] (lap + 1) << 2 | SVC_OP_* once the slot's payload is complete
    uint32_t* lens = nullptr;                           // [SVC_SLOTS] pinned, device-mapped: stored length of a run's record (AGR_CFG_VARLEN)
    uint32_t spin_cpus = 1;                             // how many waiters may spin (CPU allowance minus dispatcher and driver threads)
    std::atomic<bool> shutdown{false}, sleeping{false}; // (sleeping flips only when the ring has been empty for 2 ms)
    std::atomic<int> fatal{0};                          // a CUDA error in the dispatcher: every later call fails with it
    // ---- the words the callers / the dispatcher keep writing: a cache line each
    alignas(64) std::atomic<uint64_t> head{0};          // next ring slot to hand out (absolute number)
    alignas(64) std::atomic<uint32_t> waiters{0};       // callers blocked in svc_wait right now
    alignas(64) std::atomic<uint64_t> scanned{0};       // dispatcher: first slot whose ready word it has not consumed yet (>= taken)
    // ---- the dispatcher's own
    alignas(64) uint64_t taken = 0;                     // first slot not yet put into a batch
    uint64_t seq = 0;                                   // last batch number published
    bool running = false;                               // service kernel resident (changed under the handle mutex only)
    std::chrono::steady_clock::time_point started;      // when it was launched
    agr_k2_scratch k2{};                                // K2 scratch of the service kernel (SVC_MAX_OPS ops)
    uint32_t* d_dupfix = nullptr;
    std::atomic<uint64_t> batches{0}, ops{0};
    // diagnostics (AGR_SVC_DEBUG=1 prints them when the handle is destroyed)
    uint64_t starts = 0, stops = 0, sleeps = 0, flow_waits = 0;
    double cyc[4] = {0, 0, 0, 0}; uint64_t polls = 0;
    std::thread thr;
    alignas(64) std::mutex smu; std::condition_variable scv;   // the dispatcher sleeps here when the ring has been empty for a while
};


static void svc_fail_ops(svc_host* s, uint64_t from, uint64_t to, int rc, bool records_only);
// stops the resident kernel; the caller holds h->mu, so no new batch can be published meanwhile
static int svc_stop_locked(agr_handle* h) {
    svc_host* s = h->svc;
    if (!s || !s->running) return 0;
    s->ctl->stop = 1;
    std::atomic_thread_fence(std::memory_order_seq_cst);
    cudaError_t e = cudaStreamSynchronize(h->stream);
    s->ctl->stop = 0;
    s->running = false;
    s->stops++;
    s->cyc[0] += (double)s->ctl->cyc_wait; s->cyc[1] += (double)s->ctl->cyc_load; s->cyc[2] += (double)s->ctl->cyc_work; s->cyc[3] += (double)s->ctl->cyc_publish;
    s->polls += s->ctl->heartbeat;
    if (e != cudaSuccess) { s->fatal = AGR_ECUDA; return fail(AGR_ECUDA, std::string("service kernel: ") + cudaGetErrorString(e)); }
    if (s->ctl->done_seq != s->seq) {
        // (cannot happen while the dispatcher runs: it stops the kernel after 2 ms without traffic, the kernel's own idle exit is 2 s)
        // whoever waits for an operation of those batches gets an error instead of waiting for ever
        for (uint64_t q = s->ctl->done_seq + 1; q <= s->seq; ++q) {
            const svc_desc* dsc = s->desc + (q % SVC_DESCS);
            if (dsc->seq == q) svc_fail_ops(s, dsc->from, dsc->from + dsc->count, AGR_ECUDA, false);
        }
        s->fatal = AGR_ECUDA;
        return fail(AGR_ECUDA, "service kernel left with batches unprocessed");
    }
    return 0;
}
static int svc_start_locked(agr_handle* h) {
    svc_host* s = h->svc;
    if (s->running) return 0;
    svc_dev v{};
    v.desc = s->desc; v.payload = s->payload; v.lens = s->lens; v.res = s->res; v.ctl = s->ctl; v.dupfix = s->d_dupfix;
    v.idle_ns = 2000000000ULL;                                   // safety only: the dispatcher stops the kernel long before
    s->ctl->state = 1; s->ctl->stop = 0;
    std::atomic_thread_fence(std::memory_order_seq_cst);
    sync_window(h);
    // resume at the first batch the previous incarnation did not run (normally none is pending; a batch published right
    // before this launch is)
    cudaError_t e = agr_launch_svc(h->d, v, s->k2, s->ctl->done_seq + 1, (h->cfg.flags & AGR_CFG_VARLEN) != 0, h->stream);
    if (e != cudaSuccess) { s->fatal = AGR_ECUDA; return fail(AGR_ECUDA, std::string("service kernel launch: ") + cudaGetErrorString(e)); }
    s->running = true;
    s->starts++;
    s->ctl->cyc_wait = 0; s->ctl->cyc_load = 0; s->ctl->cyc_work = 0; s->ctl->cyc_publish = 0; s->ctl->heartbeat = 0;
    s->started = std::chrono::steady_clock::now();
    return 0;
}

// the handle lock every entry point other than the single-request path takes: the resident kernel owns the handle's stream
// while it runs, so it is stopped first (it finishes the batches already published) and started again by the dispatcher
struct HLock {
    agr_handle* h;
    explicit HLock(agr_handle* h_) : h(h_) {
        h->mu.lock();
        if (h->svc && h->svc->running) { cudaSetDevice(h->device); svc_stop_locked(h); }
    }
    ~HLock() { h->mu.unlock(); }
    HLock(const HLock&) = delete; HLock& operator=(const HLock&) = delete;
};

// answers every op of [from, to) from the host side (slab full, CUDA error): the callers see rc.  Backwards, so that the
// continuation cells of a run get their tag before its head's answer (its collector then releases every cell of the run).
static void svc_fail_ops(svc_host* s, uint64_t from, uint64_t to, int rc, bool records_only) {
    for (uint64_t a = to; a-- > from;) {
        const uint32_t slot = (uint32_t)(a & (SVC_SLOTS - 1u));
        const uint32_t rw = s->ready[slot].load(std::memory_order_relaxed), kd = rw & 3u;
        const bool rec = kd == SVC_OP_RECORD || kd == SVC_OP_CONT;
        // (a skipped slot has no waiter and keeps its old answer; it may even have been published again for the NEXT lap already)
        if ((rw >> 2) != (uint32_t)(a / SVC_SLOTS) + 1u || kd == SVC_OP_SKIP || (records_only && !rec)) continue;
        svc_res* r = s->res + slot;
        r->w[0] = rec ? 0u : (uint32_t)rc; r->w[1] = rec ? (uint32_t)rc : 0u; r->w[2] = 0;
        std::atomic_thread_fence(std::memory_order_release);
        r->w[3] = svc_tag(a) << 16;
    }
}

static void svc_dispatcher(agr_handle* h) {
    svc_host* s = h->svc;
    cudaSetDevice(h->device);
    auto last_work = std::chrono::steady_clock::now();
    uint32_t spins = 0;
    // the contiguous published prefix [taken, to), grown INCREMENTALLY: a slot is looked at until it is published and never again
    // (re-reading the callers' ready words every iteration keeps pulling their cache lines away from the cores that write them)
    uint64_t to = s->taken;
    uint32_t nrec = 0;
    uint32_t kinds[SVC_MAX_OPS / 16] = {0};
    // variable-length records: runs of slots, 128 record slots per batch (one shared-memory stage of k_svc), and their bytes
    const bool var = (h->cfg.flags & AGR_CFG_VARLEN) != 0;
    uint32_t nslots = 0;
    uint64_t nbytes = 0;
    while (!s->shutdown.load(std::memory_order_acquire)) {
        // (csrc/agr_ring.hpp: shared with the CPU simulations of the ring)
        if (var) svc_scan_run(s, s->taken, &to, &nrec, &nslots, &nbytes, kinds, 128u);
        else svc_scan(s, s->taken, &to, &nrec, kinds, 128u);
        const auto now = std::chrono::steady_clock::now();
        if (to == s->taken) {
            const auto idle = std::chrono::duration_cast<std::chrono::microseconds>(now - last_work).count();
            if (idle > 2000) {
                // nothing for 2 ms: give the GPU (and this core) back; the next caller wakes us up
                { std::lock_guard<std::mutex> hl(h->mu); if (s->running) svc_stop_locked(h); }
                std::unique_lock<std::mutex> lk(s->smu);
                s->sleeping.store(true, std::memory_order_seq_cst);
                s->sleeps++;
                const uint32_t slot = (uint32_t)(s->taken & (SVC_SLOTS - 1u));
                if ((s->ready[slot].load(std::memory_order_seq_cst) >> 2) != (uint32_t)(s->taken / SVC_SLOTS) + 1u && !s->shutdown.load())
                    s->scv.wait_for(lk, std::chrono::milliseconds(50));
                s->sleeping.store(false, std::memory_order_seq_cst);
                last_work = std::chrono::steady_clock::now();
            } else {
                cpu_relax(spins);
            }
            continue;
        }
        last_work = now;
        // Batching window = the kernel's own pace: at most two batches are outstanding (one being decided, one being pulled by
        // the kernel's loader warps); while both are, keep collecting — whatever arrives meanwhile joins the next batch instead
        // of queueing behind a train of one-request batches.
        if (s->running && s->seq - s->ctl->done_seq >= 2 && to - s->taken < SVC_MAX_OPS) {
            s->flow_waits++;
            for (int k = 0; k < 8; ++k) _mm_pause();
            continue;
        }
        spins = 0;
        std::lock_guard<std::mutex> hl(h->mu);
        if (s->fatal.load()) { svc_fail_ops(s, s->taken, to, s->fatal.load(), false); s->taken = to; nrec = 0; nslots = 0; nbytes = 0; memset(kinds, 0, sizeof kinds); continue; }
        if (s->running && s->ctl->state != 1u) {                // it left on its own (safety timeout): note it and start another
            cudaStreamSynchronize(h->stream);
            s->running = false;
        }
        // a resident kernel blocks device-wide synchronisations of other threads (cudaFree ...): let it go every 20 ms
        if (s->running && std::chrono::duration_cast<std::chrono::milliseconds>(now - s->started).count() > 20) svc_stop_locked(h);
        uint64_t first = 0, vbase = 0;
        bool have_rows = true;
        if (nrec) {
            const int rc = var ? reserve_var_locked(h, nrec, nbytes, &first, &vbase) : reserve_rows_locked(h, nrec, &first);
            if (rc < 0) { svc_fail_ops(s, s->taken, to, var ? rc : AGR_ENOSPC, true); have_rows = false; }
        }
        svc_desc dsc{};
        for (uint32_t k = 0; k < (uint32_t)(to - s->taken); ++k) {
            uint32_t kd = (kinds[k >> 4] >> ((k & 15u) * 2u)) & 3u;
            if ((kd == SVC_OP_RECORD || kd == SVC_OP_CONT) && !have_rows) kd = SVC_OP_SKIP;
            dsc.kinds[k >> 4] |= kd << ((k & 15u) * 2u);
        }
        dsc.from = s->taken; dsc.count = (uint32_t)(to - s->taken); dsc.n_records = have_rows ? nrec : 0u;
        dsc.first_l = first; dsc.first_p = (uint32_t)phys_row(h, first);
        dsc.tail = h->tail; dsc.head_l = h->rows_used; dsc.tail_phys = is_ring(h) ? (uint32_t)(h->tail % h->cfg.slab_rows) : 0u;
        dsc.idx_base = h->d.idx_base;
        dsc.vbase = vbase;
        dsc.seq = s->seq + 1;
        dsc.check = agr_svc_desc_check(&dsc);
        svc_desc* slot = s->desc + (dsc.seq % SVC_DESCS);
        // the batch number goes last; the kernel also verifies the check word, so a torn read is never accepted
        const uint64_t* src = reinterpret_cast<const uint64_t*>(&dsc);
        volatile uint64_t* dst = reinterpret_cast<volatile uint64_t*>(slot);
        for (int i = 0; i < 31; ++i) dst[i] = src[i];
        std::atomic_thread_fence(std::memory_order_release);
        dst[31] = src[31];
        std::atomic_thread_fence(std::memory_order_seq_cst);
        s->seq = dsc.seq;
        s->taken = to;
        s->batches.fetch_add(1, std::memory_order_relaxed);
        const uint32_t nops = dsc.count - (var ? nslots - nrec : 0u);   // operations (a run is one)
        s->ops.fetch_add(nops, std::memory_order_relaxed);
        h->k1_launches += nrec ? 1 : 0;                         // accounting: batches with records / with outcomes served by k_svc
        h->k2_launches += (nops > nrec) ? 1 : 0;
        nrec = 0; nslots = 0; nbytes = 0; memset(kinds, 0, sizeof kinds);
        if (!s->running && svc_start_locked(h) < 0) {
            // could not launch: nothing will ever process this batch — fail it from here
            svc_fail_ops(s, dsc.from, to, AGR_ECUDA, false);
        }
    }
    std::lock_guard<std::mutex> hl(h->mu);
    cudaSetDevice(h->device);
    svc_stop_locked(h);
}

// CPUs this process may keep busy: the cgroup CPU quota if there is one, else the online CPUs
static uint32_t cpu_allowance() {
    uint32_t n = std::max(1u, std::thread::hardware_concurrency());
    if (FILE* f = fopen("/sys/fs/cgroup/cpu.max", "r")) {
        char a[64]; unsigned long long period = 0;
        if (fscanf(f, "%63s %llu", a, &period) == 2 && strcmp(a, "max") != 0 && period) {
            const unsigned long long q = strtoull(a, nullptr, 10);
            if (q) n = std::min<uint32_t>(n, (uint32_t)std::max<unsigned long long>(1, q / period));
        }
        fclose(f);
    }
    return n;
}

static int svc_create(agr_handle* h) {
    svc_host* s = new svc_host();
    h->svc = s;
    auto pin = [&](void** p, size_t bytes) -> int {
        cudaError_t e = cudaHostAlloc(p, bytes, cudaHostAllocMapped | cudaHostAllocPortable);
        if (e != cudaSuccess) return fail(AGR_ENOMEM, std::string("cudaHostAlloc (request ring): ") + cudaGetErrorString(e));
        memset(*p, 0, bytes);
        h->host_allocs.push_back(*p);
        return 0;
    };
    TRY(pin((void**)&s->desc, sizeof(svc_desc) * SVC_DESCS));
    TRY(pin((void**)&s->payload, (size_t)SVC_SLOTS * SVC_PAYLOAD));
    TRY(pin((void**)&s->res, sizeof(svc_res) * SVC_SLOTS));
    TRY(pin((void**)&s->lens, sizeof(uint32_t) * SVC_SLOTS));
    TRY(pin((void**)&s->ctl, sizeof(svc_ctl)));
    s->ready = new std::atomic<uint32_t>[SVC_SLOTS];
    for (uint32_t i = 0; i < SVC_SLOTS; ++i) s->ready[i].store(0);
    TRY(dev_alloc(h, &s->k2.ops, (size_t)SVC_MAX_OPS, false));
    TRY(dev_alloc(h, &s->k2.nxt, (size_t)SVC_MAX_OPS, false));
    TRY(dev_alloc(h, &s->k2.eff, (size_t)SVC_MAX_OPS + 8, false));
    TRY(dev_alloc(h, &s->k2.results, (size_t)SVC_MAX_OPS, false));
    TRY(dev_alloc(h, &s->d_dupfix, (size_t)4, true));
    CK(cudaStreamSynchronize(h->stream));
    const uint32_t cpus = cpu_allowance();
    s->spin_cpus = cpus > 6 ? cpus - 6 : 1;             // leave room for the dispatcher, the driver's threads and the nappers' wake-ups
    s->thr = std::thread(svc_dispatcher, h);
    return 0;
}
static void svc_destroy(agr_handle* h) {
    svc_host* s = h->svc;
    if (!s) return;
    if (s->thr.joinable()) {
        s->shutdown.store(true, std::memory_order_release);
        { std::lock_guard<std::mutex> lk(s->smu); s->scv.notify_all(); }
        s->thr.join();
    }
    if (getenv("AGR_SVC_DEBUG")) {
        const double mhz = 1965.0, tot = s->cyc[0] + s->cyc[1] + s->cyc[2] + s->cyc[3];
        const double nb = (double)std::max<uint64_t>(1, s->batches.load());
        fprintf(stderr, "[agr svc] batches %llu ops %llu (%.1f/batch) | kernel starts %llu stops %llu, dispatcher sleeps %llu, flow waits %llu | "
                        "per batch: wait %.2f us, load %.2f us, work %.2f us, publish %.2f us (kernel alive %.1f ms), polls %llu\n",
                (unsigned long long)s->batches.load(), (unsigned long long)s->ops.load(), (double)s->ops.load() / nb,
                (unsigned long long)s->starts, (unsigned long long)s->stops, (unsigned long long)s->sleeps, (unsigned long long)s->flow_waits,
                s->cyc[0] / mhz / nb, s->cyc[1] / mhz / nb, s->cyc[2] / mhz / nb, s->cyc[3] / mhz / nb, tot / mhz / 1000.0, (unsigned long long)s->polls);
    }
    delete[] s->ready;
    h->svc = nullptr;
    delete s;
}

// (the callers' side of the ring — svc_submit_one, svc_try, svc_wait, svc_release — is csrc/agr_ring.hpp: the same code runs against a
// stand-in for the dispatcher and the GPU in tests/ring_sim.cpp, on the CPU)
// Request.ID of the record in ring slot a: minted from its row, or the caller's own (still in the slot's payload)
static inline void svc_request_id(agr_handle* h, uint64_t a, uint64_t rid, uint8_t id[16]) {
    if (h->cfg.flags & AGR_CFG_MINT_IDS) {
        unsigned long long lo, hi;
        agr_mint_id(rid, h->d.shard_id, h->d.id_gen, h->d.id_secret, lo, hi);
        memcpy(id, &lo, 8); memcpy(id + 8, &hi, 8);
    } else memcpy(id, h->svc->payload + (size_t)(a & (SVC_SLOTS - 1u)) * SVC_PAYLOAD, 16);
}

static int svc_ingest(agr_handle* h, const agr_record* recs, uint32_t n, agr_verdict* out, uint8_t (*ids)[16], uint64_t* first_rid) {
    svc_host* s = h->svc;
    uint64_t pos[SVC_MAX_CALL];
    for (uint32_t i = 0; i < n; ++i) while (!svc_submit_one(s, SVC_OP_RECORD, &recs[i], sizeof(agr_record), &pos[i])) {}   // in call order
    int rc = 0;
    for (uint32_t i = 0; i < n; ++i) {
        svc_answer r; svc_wait(s, pos[i], &r);
        if ((r.w0 & 0xffu) == 0u) rc = (int)r.w1;
        else {
            if (out) { memcpy(&out[i], &r.w0, 4); memcpy((uint8_t*)&out[i] + 4, &r.w1, 4); }
            if (ids) svc_request_id(h, pos[i], r.rid, ids[i]);
            if (i == 0 && first_rid) *first_rid = r.rid;
        }
        svc_release(s, pos[i]);
    }
    if (rc < 0) return fail(rc, rc == AGR_ENOSPC ? "slab full" : "single-request front end: CUDA error");
    return 0;
}
static int svc_complete(agr_handle* h, const agr_outcome* outs, uint32_t n, int32_t* results) {
    svc_host* s = h->svc;
    uint64_t pos[SVC_MAX_CALL];
    for (uint32_t i = 0; i < n; ++i) while (!svc_submit_one(s, SVC_OP_OUTCOME, &outs[i], sizeof(agr_outcome), &pos[i])) {}
    int rc = 0;
    for (uint32_t i = 0; i < n; ++i) {
        svc_answer r; svc_wait(s, pos[i], &r);
        const int32_t res = (int32_t)r.w0;
        if (res < 0 && res != AGR_ENOTFOUND) rc = res;
        if (results) results[i] = res;
        svc_release(s, pos[i]);
    }
    if (rc < 0) return fail(rc, "single-request front end: CUDA error");
    return 0;
}
// variable-length records (offsets already checked): one run of slots per record, in call order
static int svc_ingest_var(agr_handle* h, const uint8_t* blob, const uint32_t* offsets, uint32_t n, agr_verdict* out, uint8_t (*ids)[16],
                          uint64_t* first_rid) {
    svc_host* s = h->svc;
    uint64_t pos[SVC_MAX_CALL];
    for (uint32_t i = 0; i < n; ++i)
        while (!svc_submit_run(s, blob + offsets[i], offsets[i + 1] - offsets[i], &pos[i])) {}    // a run not free: draw again
    int rc = 0;
    for (uint32_t i = 0; i < n; ++i) {
        svc_answer r; svc_wait(s, pos[i], &r);
        if ((r.w0 & 0xffu) == 0u) rc = (int)r.w1;
        else {
            if (out) { memcpy(&out[i], &r.w0, 4); memcpy((uint8_t*)&out[i] + 4, &r.w1, 4); }
            if (ids) svc_request_id(h, pos[i], r.rid, ids[i]);
            if (i == 0 && first_rid) *first_rid = r.rid;
        }
        svc_release_run(s, pos[i], svc_run_slots(offsets[i + 1] - offsets[i]));
    }
    if (rc < 0) return fail(rc, rc == AGR_ENOSPC ? "byte slab or slab full" : rc == AGR_EINVAL ? "batch larger than half the byte slab" : "single-request front end: CUDA error");
    return 0;
}

extern "C" {

uint32_t agr_abi_version(void) { return AGR_ABI_VERSION; }
const char* agr_last_error(void) { return g_err.c_str(); }
const char* agr_strerror(int code) {
    switch (code) {
        case AGR_OK: return "ok";
        case AGR_EINVAL: return "invalid argument";
        case AGR_ENODEV: return "no usable CUDA device";
        case AGR_ENOMEM: return "out of memory";
        case AGR_ENOSPC: return "capacity exhausted";
        case AGR_ENOTFOUND: return "not found";
        case AGR_ECUDA: return "CUDA error";
        case AGR_ECAP: return "output array too small";
        case AGR_ECOMM: return "multi-GPU exchange error";
        default: return "unknown error";
    }
}

void* agr_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { g_err = "cudaHostAlloc failed"; return nullptr; }
    return p;
}
void agr_host_free(void* p) { if (p) cudaFreeHost(p); }

static int create_impl(const agr_config* cfg_in, agr_handle* h) {
    agr_config c{};
    if (cfg_in) c = *cfg_in;
    if (c.flags == 0) c.flags = AGR_CFG_PERSISTENCE;
    if (c.slab_rows == 0) c.slab_rows = 1ull << 20;
    if (c.slab_rows >= 0x7fffffffull) return fail(AGR_EINVAL, "slab_rows must be < 2^31");
    const bool mint = (c.flags & AGR_CFG_MINT_IDS) != 0;
    if (mint) c.table_slots = 64;                               // no dedupe index in this mode (a stub keeps pointers valid)
    if (c.table_slots == 0) c.table_slots = next_pow2(c.slab_rows * 2);
    if (c.table_slots & (c.table_slots - 1)) return fail(AGR_EINVAL, "table_slots must be a power of two");
    if (!mint && c.table_slots < c.slab_rows + c.slab_rows / 4) return fail(AGR_EINVAL, "table_slots must be >= 1.25 * slab_rows");
    if (c.table_slots > (1ull << 32)) return fail(AGR_EINVAL, "table_slots must be <= 2^32");
    if (c.max_agents == 0) c.max_agents = 4096;
    if (c.max_agents >= RT_SLOT_NONE) return fail(AGR_EINVAL, "max_agents must be < 2^23 - 1");
    if (c.max_batch == 0) c.max_batch = 1u << 20;
    if (c.flags & AGR_CFG_RING) {
        if (c.max_batch > c.slab_rows / 2) c.max_batch = (uint32_t)(c.slab_rows / 2);
        if (c.max_batch == 0) return fail(AGR_EINVAL, "AGR_CFG_RING: slab_rows too small");
    }
    if (c.log_entries == 0) c.log_entries = c.slab_rows * 3;   // a replayed request pushes twice (Q7), plus once per earlier retry
    if ((c.k1_variant & 0xfu) == 0) c.k1_variant |= 4u;      // default K1 shape: TMA, 14 warps x 1 stage, fused index
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(AGR_ENODEV, "no CUDA device visible (this library has no CPU fallback)"); }
    int dev = c.device;
    if (dev < 0) { if (cudaGetDevice(&dev) != cudaSuccess) return fail(AGR_ENODEV, "cudaGetDevice failed"); }
    if (dev >= ndev) return fail(AGR_ENODEV, "device ordinal out of range");
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, dev));
    if (prop.major < 10) return fail(AGR_ENODEV, std::string("device ") + prop.name + " is sm_" + std::to_string(prop.major * 10 + prop.minor) + "; this library is built for sm_100a only");
    CK(cudaSetDevice(dev));
    h->device = dev;
    h->sm_count = prop.multiProcessorCount;
    h->cfg = c;
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->d2h_stream, cudaStreamNonBlocking));
    agr_dev& d = h->d;
    const bool varlen = (c.flags & AGR_CFG_VARLEN) != 0;
    if (varlen) {
        if (c.vslab_bytes == 0) c.vslab_bytes = 1024ull * c.slab_rows;
        h->cfg = c;
        h->vcap = c.vslab_bytes;
        TRY(dev_alloc(h, &d.slab, (size_t)c.vslab_bytes + AGR_VT_MAXREC, false));
        TRY(dev_alloc(h, &d.voff, c.slab_rows, true));
        TRY(dev_alloc(h, &d.vlen, c.slab_rows, true));
        TRY(dev_alloc(h, &h->d_voffsets, (size_t)c.max_batch + 1, false));
        TRY(host_alloc(h, &h->h_voffsets, (size_t)c.max_batch + 1));
        TRY(dev_alloc(h, &h->d_tile_first, (size_t)(((size_t)c.max_batch * AGR_VT_MAXREC) / AGR_VT_TILE + 8), false));
    } else {
        TRY(dev_alloc(h, &d.slab, (size_t)c.slab_rows * AGR_REC, false));
    }
    TRY(dev_alloc(h, &d.state, c.slab_rows + 4, true));        // (+4: k3_mark reads these two four rows at a time)
    TRY(dev_alloc(h, &d.route, c.slab_rows + 4, true));
    TRY(dev_alloc(h, &d.aux, c.slab_rows, true));
    TRY(dev_alloc(h, &d.cksum, c.slab_rows, true));
    TRY(dev_alloc(h, &d.table, c.table_slots, true));
    d.table_mask = c.table_slots - 1;
    uint32_t acap = (uint32_t)next_pow2((uint64_t)c.max_agents * 2);
    TRY(dev_alloc(h, &d.akeys, acap, true));
    d.amask = acap - 1;
    h->akeys_host.assign(acap, agr_agent_key{});
    TRY(dev_alloc(h, &d.astatus, c.max_agents, true));
    TRY(dev_alloc(h, &d.ctr, (size_t)C_NCTR, true));
    TRY(dev_alloc(h, &d.completed_log, c.log_entries, false));
    TRY(dev_alloc(h, &d.failed_log, c.log_entries, false));
    TRY(dev_alloc(h, &d.log_len, (size_t)2, true));
    d.log_cap = c.log_entries;
    TRY(dev_alloc(h, &d.marks, (size_t)(2 * (size_t)c.max_batch / 32 + 8), true));   // (2 x max_batch: the exchange runs K1 over own + received rows)
    TRY(dev_alloc(h, &d.dupfix, (size_t)8, true));
    h->dupfix_base = d.dupfix; d.dupfix_next = d.dupfix + 4;
    if (c.flags & AGR_CFG_RING) {
        TRY(dev_alloc(h, &h->d_log_scratch, c.log_entries, false));
        TRY(dev_alloc(h, &h->d_lc_chunks, (size_t)(c.log_entries / 1024 + 4), false));
    }
    if (c.resp_bytes == 0) c.resp_bytes = 64ull * c.slab_rows;
    h->cfg.resp_bytes = c.resp_bytes; h->resp_cap = c.resp_bytes;
    TRY(dev_alloc(h, &h->d_resp, (size_t)c.resp_bytes, false));
    TRY(dev_alloc(h, &h->d_resp_off, c.slab_rows, true));
    TRY(dev_alloc(h, &h->d_resp_len, c.slab_rows, true));
    TRY(dev_alloc(h, &h->d_resp_hlen, c.slab_rows, true));
    TRY(dev_alloc(h, &h->d_err_off, c.slab_rows, true));
    TRY(dev_alloc(h, &h->d_err_len, c.slab_rows, true));
    TRY(dev_alloc(h, &d.ptime, c.slab_rows, true));
    TRY(dev_alloc(h, &d.mtime, c.slab_rows, true));
    TRY(dev_alloc(h, &d.head, c.slab_rows, true));
    TRY(dev_alloc(h, &d.cmin, (size_t)(c.slab_rows / AGR_CHUNK_ROWS + 2), false));
    CK(cudaMemsetAsync(d.cmin, 0xff, (size_t)(c.slab_rows / AGR_CHUNK_ROWS + 2) * 8, h->stream));   // ~0: no stored row in any chunk yet
    // the key of the id permutation: drawn from the OS CSPRNG unless the caller brings one (a restore passes the snapshot's),
    // so that ids of one engine instance never resolve in another and cannot be guessed (the reference mints uuid.New())
    d.id_secret = c.id_secret;
    while (d.id_secret == 0) {
        if (getrandom(&d.id_secret, sizeof d.id_secret, 0) != (ssize_t)sizeof d.id_secret) return fail(AGR_EINVAL, "getrandom failed: pass agr_config.id_secret");
    }
    h->cfg.id_secret = d.id_secret;
    d.shard_id = 0; d.id_gen = 1; d.tail = 0; d.head_l = 0; d.ring_rows = 0; d.tail_phys = 0; d.idx_base = 0;
    if (!varlen && (c.k1_variant & 0xfu) != AGR_K1_LSU && agr_k1_tma_make_map(d.slab, c.slab_rows, h->tmap) != 0)
        return fail(AGR_ECUDA, "cuTensorMapEncodeTiled failed for the slab");
    d.cfg_flags = c.flags & 0xffffu;
    if (c.k1_variant & 0x10u) d.cfg_flags |= AGR_CFGI_SPLIT_INDEX;
    // staging
    h->bounce_bytes = std::min<size_t>((size_t)c.max_batch * AGR_REC, (size_t)32 << 20);
    for (int k = 0; k < 2; ++k) {
        TRY(host_alloc(h, &h->bounce[k], h->bounce_bytes));
        CK(cudaEventCreateWithFlags(&h->bounce_ev[k], cudaEventDisableTiming));
    }
    TRY(host_alloc(h, &h->h_verdicts, c.max_batch));
    TRY(dev_alloc(h, &h->d_verdicts, c.max_batch, false));
    TRY(dev_alloc(h, &h->d_ids, (size_t)c.max_batch * 16, false));
    TRY(host_alloc(h, &h->h_ids, (size_t)c.max_batch * 16));
    TRY(host_alloc(h, &h->h_ops, (size_t)16));
    TRY(host_alloc(h, &h->h_outs, c.max_batch));
    TRY(dev_alloc(h, &h->d_outs, c.max_batch, false));
    TRY(host_alloc(h, &h->h_results, c.max_batch));
    TRY(host_alloc(h, &h->h_small, (size_t)64));
    TRY(dev_alloc(h, &h->d_reclaim, (size_t)64, true));
    TRY(dev_alloc(h, &h->d_reclaim_scratch, (size_t)2, false));
    { const uint32_t init[2] = {0xffffffffu, 0u}; CK(cudaMemcpyAsync(h->d_reclaim_scratch, init, 8, cudaMemcpyHostToDevice, h->stream)); CK(cudaStreamSynchronize(h->stream)); }
    TRY(host_alloc(h, &h->h_reclaim, (size_t)64));
    TRY(dev_alloc(h, &h->d_ops, (size_t)16, false));
    TRY(dev_alloc(h, &h->d_hrid, (size_t)16, false));
    TRY(host_alloc(h, &h->h_k2flag, (size_t)4));
    TRY(k2_scratch_alloc(h, c.max_batch));
    TRY(dev_alloc(h, &h->d_gtotal, ((size_t)c.max_agents + 8) * 66, false));   // gtotal + 64 segment partials per group
    TRY(dev_alloc(h, &h->d_goff, (size_t)c.max_agents + 2, false));
    TRY(dev_alloc(h, &h->d_min_inq, (size_t)1, false));
    CK(cudaStreamSynchronize(h->stream));
    if (c.flags & AGR_CFG_COMBINE) TRY(svc_create(h));
    return 0;
}

int agr_create(const agr_config* cfg, agr_handle** out) {
    if (!out) return fail(AGR_EINVAL, "out is NULL");
    *out = nullptr;
    agr_handle* h = new agr_handle();
    int r = create_impl(cfg, h);
    if (r < 0) { std::string keep = g_err; agr_destroy(h); g_err = keep; return r; }
    *out = h;
    return 0;
}

void agr_destroy(agr_handle* h) {
    if (!h) return;
    svc_destroy(h);
    if (h->stream) { cudaSetDevice(h->device); cudaStreamSynchronize(h->stream); }
    for (void* p : h->dev_allocs) cudaFree(p);
    for (void* p : h->host_allocs) cudaFreeHost(p);
    for (int k = 0; k < 2; ++k) if (h->bounce_ev[k]) cudaEventDestroy(h->bounce_ev[k]);
    for (auto e : h->tev) cudaEventDestroy(e);
    for (auto e : h->op_ev) if (e) cudaEventDestroy(e);
    for (auto e : h->chunk_ev) cudaEventDestroy(e);
    if (h->reclaim_ev) cudaEventDestroy(h->reclaim_ev);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->d2h_stream) cudaStreamDestroy(h->d2h_stream);
    for (auto e : h->out_ev) cudaEventDestroy(e);
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

// ------------------------------------------------------------------------------------------ agent table
static int agent_find(agr_handle* h, const char* id) {
    auto it = h->slot_of.find(std::string(id));
    return it == h->slot_of.end() ? -1 : (int)it->second;
}

// status lives in two places on the device: astatus[slot] (K3 reads it by slot) and the key entry (K1 reads it with
// the key in one access); both copies are stream-ordered before the next kernel
static int push_agent_status(agr_handle* h, uint32_t slot, uint8_t status) {
    const uint32_t idx = h->akey_index[slot];
    h->akeys_host[idx].status = status;
    CK(cudaMemcpyAsync(h->d.astatus + slot, &status, 1, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(&h->d.akeys[idx].status, &h->akeys_host[idx].status, 4, cudaMemcpyHostToDevice, h->stream));
    return 0;
}

// core of agr_set_agent_state; `upload` = push the change to the device now (the bulk call uploads the tables once instead)
static int set_agent_state_locked(agr_handle* h, const char* agent_id, uint8_t status, bool upload) {
    size_t len = strnlen(agent_id, AGR_AGENT_ID_BYTES);
    if (len == 0 || len >= AGR_AGENT_ID_BYTES) return fail(AGR_EINVAL, "agent id must be 1..31 bytes");
    if (status > AGR_AGENT_FAILED) return fail(AGR_EINVAL, "bad agent status");
    int slot = agent_find(h, agent_id);
    if (slot < 0) {
        if (h->agent_names.size() >= h->cfg.max_agents) return fail(AGR_ENOSPC, "agent table full");
        slot = (int)h->agent_names.size();
        h->agent_names.emplace_back(agent_id);
        h->agent_status.push_back(status);
        h->slot_of.emplace(std::string(agent_id), (uint32_t)slot);
        agr_agent_key key{};
        pack_agent_id(agent_id, key.w);
        key.slot = (uint32_t)slot;
        key.status = status;
        uint32_t idx = (uint32_t)agr_hash_agent(key.w[0], key.w[1], key.w[2], key.w[3]) & h->d.amask;
        while (h->akeys_host[idx].w[0] | h->akeys_host[idx].w[1] | h->akeys_host[idx].w[2] | h->akeys_host[idx].w[3])
            idx = (idx + 1) & h->d.amask;
        h->akeys_host[idx] = key;
        h->akey_index.push_back(idx);
        if (upload) {
            // status first, then the key that makes the slot reachable; both are stream-ordered before the next kernel
            CK(cudaMemcpyAsync(h->d.astatus + slot, &status, 1, cudaMemcpyHostToDevice, h->stream));
            CK(cudaMemcpyAsync(h->d.akeys + idx, &key, sizeof key, cudaMemcpyHostToDevice, h->stream));
        }
    } else {
        h->agent_status[slot] = status;
        if (upload) TRY(push_agent_status(h, (uint32_t)slot, status));
        else h->akeys_host[h->akey_index[slot]].status = status;
    }
    return slot;
}
int agr_set_agent_state(agr_handle* h, const char* agent_id, uint8_t status) {
    if (!h || !agent_id) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    return set_agent_state_locked(h, agent_id, status, true);
}
int agr_set_agent_states(agr_handle* h, const char (*agent_ids)[AGR_AGENT_ID_BYTES], const uint8_t* statuses, uint32_t n, int32_t* slots) {
    if (!h || (n && (!agent_ids || !statuses))) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    const bool bulk = n > 16;                       // many writes: update the host mirror, upload both tables once
    int rc = 0;
    for (uint32_t i = 0; i < n; ++i) {
        char id[AGR_AGENT_ID_BYTES];
        memcpy(id, agent_ids[i], AGR_AGENT_ID_BYTES); id[AGR_AGENT_ID_BYTES - 1] = 0;
        const int s = set_agent_state_locked(h, id, statuses[i], !bulk);
        if (slots) slots[i] = s;
        if (s < 0 && rc == 0) rc = s;               // keep going: one bad entry must not hide the other status writes
    }
    if (bulk && !h->agent_status.empty()) {
        CK(cudaMemcpyAsync(h->d.astatus, h->agent_status.data(), h->agent_status.size(), cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->d.akeys, h->akeys_host.data(), h->akeys_host.size() * sizeof(agr_agent_key), cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));       // the host vectors may be reallocated by the next call
    }
    return rc;
}

int agr_agent_slot(agr_handle* h, const char* agent_id) {
    if (!h || !agent_id) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    int s = agent_find(h, agent_id);
    if (s < 0 || h->agent_status[s] == AG_STATUS_REMOVED) return fail(AGR_ENOTFOUND, "agent not found");
    return s;
}

int agr_drop_agent(agr_handle* h, const char* agent_id) {
    if (!h || !agent_id) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    int slot = agent_find(h, agent_id);
    if (slot < 0) return fail(AGR_ENOTFOUND, "agent not found");
    h->agent_status[slot] = AG_STATUS_REMOVED;
    TRY(push_agent_status(h, (uint32_t)slot, AG_STATUS_REMOVED));                          // DEL agent:{id} (agent.go:344)
    unsigned long long lens[2];
    CK(cudaMemcpyAsync(lens, h->d.log_len, sizeof lens, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    agr_launch_drop_agent(h->d, (uint32_t)slot, rows_span(h), std::max(lens[0], lens[1]), h->stream);
    h->k3_launches += 2;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// Rows handed out by agr_reserve_rows hold no record until agr_ingest_rows has run over them.  The replay scan, the pending
// views and agr_reclaim stop at the first such row: otherwise a scan that finds "nothing pending" above its low-water mark
// would move the mark past rows that K1 fills in later, and those requests would never be replayed.
static uint64_t ingested_bound(const agr_handle* h) {
    uint64_t b = h->rows_used;
    for (const auto& r : h->resv) b = std::min(b, r.first);
    return b;
}
static void resv_remove(agr_handle* h, uint64_t first, uint64_t end) {
    std::vector<std::pair<uint64_t, uint64_t>> keep;
    for (const auto& r : h->resv) {
        if (r.second <= first || r.first >= end) { keep.push_back(r); continue; }
        if (r.first < first) keep.emplace_back(r.first, first);
        if (r.second > end) keep.emplace_back(end, r.second);
    }
    h->resv.swap(keep);
}
// ------------------------------------------------------------------------------------------ K1
static int reserve_rows_locked(agr_handle* h, uint32_t n, uint64_t* first) {
    if (!is_ring(h)) {
        if (h->rows_used + n > h->cfg.slab_rows) return fail(AGR_ENOSPC, "slab full");
        *first = h->rows_used;
        h->rows_used += n;
        sync_window(h);
        return 0;
    }
    // ring: a batch never wraps — if it does not fit before the end of the slab, the rows up to the end are skipped
    // (they stay "no record": released rows are zeroed), at most max_batch rows per lap
    const uint64_t R = h->cfg.slab_rows;
    const uint64_t at = h->rows_used % R;
    const uint64_t pad = (at + n > R) ? R - at : 0;
    if (h->rows_used + pad + n - h->tail > R) return fail(AGR_ENOSPC, "slab full: agr_expire + agr_reclaim release rows at the tail");
    h->rows_used += pad;
    *first = h->rows_used;
    h->rows_used += n;
    sync_window(h);
    return 0;
}

// every K1 batch gets a zeroed set of per-batch words; the set it does not use is cleared by its k1_post for the next one
static inline void flip_batch_words(agr_handle* h) {
    h->batch_phase ^= 1u;
    h->d.dupfix = h->dupfix_base + 4u * h->batch_phase;
    h->d.dupfix_next = h->dupfix_base + 4u * (h->batch_phase ^ 1u);
}
static int launch_k1_locked(agr_handle* h, uint64_t first, uint32_t n, agr_verdict* d_out, uint8_t* d_ids = nullptr) {
    sync_window(h);
    flip_batch_words(h);
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    // AGR_CFG_TIMING: events around the K1 kernel of every launch, or of every k-th one (k1_variant bits 16..23): an event record
    // is a stream operation of its own between two kernels, and two of them per step cost a back-to-back loop a few microseconds
    const uint32_t tstride = std::max<uint32_t>(1u, (h->cfg.k1_variant >> 16) & 0xffu);
    if ((h->cfg.flags & AGR_CFG_TIMING) && (h->timing_calls++ % tstride) == 0) {
        if (h->tev.empty()) {
            h->tev.resize(2 * AGR_TIMING_RING);
            for (auto& e : h->tev) CK(cudaEventCreate(&e));
        }
        const uint64_t k = h->tev_next++ % AGR_TIMING_RING;
        e0 = h->tev[2 * k]; e1 = h->tev[2 * k + 1];
    }
    agr_launch_k1(h->d, (uint32_t)phys_row(h, first), n, h->cfg.k1_variant, (h->cfg.k1_variant & 0xfu) != AGR_K1_LSU ? h->tmap : nullptr,
                  h->sm_count, h->stream, e0, e1, d_out, d_ids);
    h->k1_launches += agr_k1_launches_per_batch(h->cfg.k1_variant);
    CK(cudaGetLastError());
    return 0;
}

static int ingest_rows_locked(agr_handle* h, uint64_t first, uint32_t n, agr_verdict* out, bool sync) {
    if (first + n > h->rows_used) return fail(AGR_EINVAL, "rows not reserved");
    if (n > h->cfg.max_batch) return fail(AGR_EINVAL, "n exceeds max_batch");
    if (n == 0) return 0;
    TRY(launch_k1_locked(h, first, n, out ? h->d_verdicts : nullptr));
    if (!h->resv.empty()) resv_remove(h, first, first + n);
    if (out) {
        CK(cudaMemcpyAsync(h->h_verdicts, h->d_verdicts, (size_t)n * sizeof(agr_verdict), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        memcpy(out, h->h_verdicts, (size_t)n * sizeof(agr_verdict));
    } else if (sync) {
        CK(cudaStreamSynchronize(h->stream));
    }
    return 0;
}

int agr_mint_ids(agr_handle* h, uint64_t first_rid, uint32_t n, uint8_t (*ids)[16]) {
    if (!h || (n && !ids)) return fail(AGR_EINVAL, "NULL argument");
    if (!(h->cfg.flags & AGR_CFG_MINT_IDS)) return fail(AGR_EINVAL, "engine was not created with AGR_CFG_MINT_IDS");
    for (uint32_t i = 0; i < n; ++i) {
        unsigned long long lo, hi;
        agr_mint_id(first_rid + i, h->d.shard_id, h->d.id_gen, h->d.id_secret, lo, hi);
        memcpy(ids[i], &lo, 8); memcpy(ids[i] + 8, &hi, 8);
    }
    return 0;
}

int agr_reserve_rows(agr_handle* h, uint32_t n, uint64_t* first_rid) {
    if (!h || !first_rid) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    TRY(reserve_rows_locked(h, n, first_rid));
    if (n) {
        if (!h->resv.empty() && h->resv.back().second == *first_rid) h->resv.back().second += n;   // back-to-back reservations merge
        else h->resv.emplace_back(*first_rid, *first_rid + n);
    }
    return 0;
}
int agr_fill_rows(agr_handle* h, uint64_t first_rid, const agr_record* recs, uint32_t n) {
    if (!h || (n && !recs)) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    if (h->cfg.flags & AGR_CFG_VARLEN) return fail(AGR_EINVAL, "fixed-stride engines only");
    if (first_rid + n > h->rows_used || first_rid < h->tail) return fail(AGR_EINVAL, "rows not reserved");
    if (n == 0) return 0;
    if (phys_row(h, first_rid) + n > h->cfg.slab_rows) return fail(AGR_EINVAL, "row range wraps");
    CK(cudaMemcpyAsync(h->d.slab + phys_row(h, first_rid) * AGR_REC, recs, (size_t)n * AGR_REC, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}
int agr_ingest_rows(agr_handle* h, uint64_t first_rid, uint32_t n, agr_verdict* out) {
    if (!h) return fail(AGR_EINVAL, "NULL handle");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    return ingest_rows_locked(h, first_rid, n, out, true);
}
int agr_ingest_rows_async(agr_handle* h, uint64_t first_rid, uint32_t n) {
    if (!h) return fail(AGR_EINVAL, "NULL handle");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    return ingest_rows_locked(h, first_rid, n, nullptr, false);
}
int agr_sync(agr_handle* h) {
    if (!h) return fail(AGR_EINVAL, "NULL handle");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}
void* agr_stream(agr_handle* h) { return h ? (void*)h->stream : nullptr; }
void* agr_slab_ptr(agr_handle* h, uint64_t rid) {
    if (!h || rid >= h->rows_used || rid < h->tail) return nullptr;
    return (void*)(h->d.slab + phys_row(h, rid) * AGR_REC);
}

// host -> slab rows -> K1 -> verdicts, pipelined in chunks: the H2D copy of chunk k+1 (copy stream) overlaps K1 and the
// verdict D2H of chunk k (compute stream).  Chunks are consecutive sub-batches in arrival order, so the result is
// identical to one big batch (tests/test_parity_gpu.py::test_result_does_not_depend_on_batching).
// Pinned (or registered) caller memory is DMA'd in place; pageable memory goes through two pinned bounce buffers.
#define AGR_INGEST_CHUNK (1u << 17)   // 128 Ki records = 64 MiB per H2D chunk
int agr_ingest(agr_handle* h, const agr_record* recs, uint32_t n, agr_verdict* out, uint64_t* first_rid) {
    return agr_ingest_ex(h, recs, n, out, nullptr, first_rid);
}

static int ingest_ex_locked(agr_handle* h, const agr_record* recs, uint32_t n, agr_verdict* out, uint8_t (*ids)[16], uint64_t* first_rid);

int agr_ingest_ex(agr_handle* h, const agr_record* recs, uint32_t n, agr_verdict* out, uint8_t (*ids)[16], uint64_t* first_rid) {
    if (!h || (n && !recs)) return fail(AGR_EINVAL, "NULL argument");
    if (h->cfg.flags & AGR_CFG_VARLEN) return fail(AGR_EINVAL, "variable-length engine: use agr_ingest_var");
    if (h->svc && n >= 1 && n <= SVC_MAX_CALL) return svc_ingest(h, recs, n, out, ids, first_rid);
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    return ingest_ex_locked(h, recs, n, out, ids, first_rid);
}

static int ingest_ex_locked(agr_handle* h, const agr_record* recs, uint32_t n, agr_verdict* out, uint8_t (*ids)[16], uint64_t* first_rid) {
    if (n > h->cfg.max_batch) return fail(AGR_EINVAL, "n exceeds max_batch");
    uint64_t first = 0;
    TRY(reserve_rows_locked(h, n, &first));
    if (first_rid) *first_rid = first;
    if (n == 0) return 0;
    const bool src_pinned = is_pinned(recs);
    const bool out_pinned = out && is_pinned(out);
    const bool ids_pinned = ids && is_pinned(ids);
    const uint32_t nchunks = (n + AGR_INGEST_CHUNK - 1) / AGR_INGEST_CHUNK;
    while (h->chunk_ev.size() < nchunks + 1) {
        cudaEvent_t e; CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        h->chunk_ev.push_back(e);
    }
    // the copy stream must not overwrite rows before earlier work on the compute stream is done with the slab
    CK(cudaEventRecord(h->chunk_ev[nchunks], h->stream));
    CK(cudaStreamWaitEvent(h->copy_stream, h->chunk_ev[nchunks], 0));
    int bk = 0;
    for (uint32_t c = 0; c < nchunks; ++c) {
        const uint32_t off = c * AGR_INGEST_CHUNK, cn = std::min(AGR_INGEST_CHUNK, n - off);
        uint8_t* dst = h->d.slab + (phys_row(h, first) + off) * AGR_REC;
        const uint8_t* src = (const uint8_t*)(recs + off);
        size_t bytes = (size_t)cn * AGR_REC;
        if (src_pinned) {
            CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, h->copy_stream));
        } else {
            for (size_t o = 0; o < bytes;) {
                size_t piece = std::min(h->bounce_bytes, bytes - o);
                CK(cudaEventSynchronize(h->bounce_ev[bk]));
                par_memcpy(h->bounce[bk], src + o, piece);
                CK(cudaMemcpyAsync(dst + o, h->bounce[bk], piece, cudaMemcpyHostToDevice, h->copy_stream));
                CK(cudaEventRecord(h->bounce_ev[bk], h->copy_stream));
                o += piece; bk ^= 1;
            }
        }
        CK(cudaEventRecord(h->chunk_ev[c], h->copy_stream));
        CK(cudaStreamWaitEvent(h->stream, h->chunk_ev[c], 0));
        TRY(launch_k1_locked(h, first + off, cn, out ? h->d_verdicts + off : nullptr, ids ? h->d_ids + (size_t)off * 16 : nullptr));
        if (out || ids) {
            // the chunk's read-backs (8 + 16 B per record) leave on their own stream as soon as its K1 is done
            while (h->out_ev.size() <= c) { cudaEvent_t e; CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); h->out_ev.push_back(e); }
            CK(cudaEventRecord(h->out_ev[c], h->stream));
            CK(cudaStreamWaitEvent(h->d2h_stream, h->out_ev[c], 0));
            if (out) CK(cudaMemcpyAsync((out_pinned ? out : h->h_verdicts) + off, h->d_verdicts + off, (size_t)cn * sizeof(agr_verdict), cudaMemcpyDeviceToHost, h->d2h_stream));
            if (ids) CK(cudaMemcpyAsync((ids_pinned ? (uint8_t*)ids : h->h_ids) + (size_t)off * 16, h->d_ids + (size_t)off * 16, (size_t)cn * 16, cudaMemcpyDeviceToHost, h->d2h_stream));
        }
    }
    CK(cudaStreamSynchronize(h->stream));
    if (out || ids) CK(cudaStreamSynchronize(h->d2h_stream));
    if (out && !out_pinned) memcpy(out, h->h_verdicts, (size_t)n * sizeof(agr_verdict));
    if (ids && !ids_pinned) memcpy(ids, h->h_ids, (size_t)n * 16);
    return 0;
}

// ------------------------------------------------------------------------------------------ tickets (submit / collect)
uint32_t agr_ring_capacity(void) { return SVC_SLOTS; }
#define TICKET_OUTCOME (1ULL << 63)                               // a ticket = ring slot number | kind | (run length - 1) << 59
#define TICKET_RUN_SHIFT 59
#define TICKET_SLOT ((1ULL << TICKET_RUN_SHIFT) - 1ULL)
static int submit_one(agr_handle* h, uint32_t kind, const void* item, size_t bytes, agr_ticket* ticket) {
    if (!h || !item || !ticket) return fail(AGR_EINVAL, "NULL argument");
    svc_host* s = h->svc;
    if (!s) return fail(AGR_EINVAL, "engine was not created with AGR_CFG_COMBINE");
    uint64_t a = 0;
    if (!svc_submit_one(s, kind, item, bytes, &a)) return AGR_EAGAIN;   // collect outstanding tickets (agr_poll) and come again
    *ticket = a | (kind == SVC_OP_OUTCOME ? TICKET_OUTCOME : 0ULL);
    return 0;
}
int agr_submit_ingest(agr_handle* h, const agr_record* rec, agr_ticket* ticket) {
    if (h && (h->cfg.flags & AGR_CFG_VARLEN)) return fail(AGR_EINVAL, "variable-length engine: use agr_submit_ingest_var");
    return submit_one(h, SVC_OP_RECORD, rec, sizeof(agr_record), ticket);
}
static bool var_len_ok(uint32_t len) { return !(len & 15u) && len >= AGR_HEADER_BYTES && len <= AGR_VAR_MAX_RECORD; }
int agr_submit_ingest_var(agr_handle* h, const uint8_t* rec, uint32_t len, agr_ticket* ticket) {
    if (!h || !rec || !ticket) return fail(AGR_EINVAL, "NULL argument");
    if (!(h->cfg.flags & AGR_CFG_VARLEN)) return fail(AGR_EINVAL, "engine was not created with AGR_CFG_VARLEN");
    svc_host* s = h->svc;
    if (!s) return fail(AGR_EINVAL, "engine was not created with AGR_CFG_COMBINE");
    if (!var_len_ok(len)) return fail(AGR_EINVAL, "record length must be a multiple of 16 in [96, 8192]");
    uint64_t a = 0;
    if (!svc_submit_run(s, rec, len, &a)) return AGR_EAGAIN;            // collect outstanding tickets (agr_poll) and come again
    *ticket = a | (uint64_t)(svc_run_slots(len) - 1u) << TICKET_RUN_SHIFT;
    return 0;
}
int agr_submit_complete(agr_handle* h, const agr_outcome* outcome, agr_ticket* ticket) { return submit_one(h, SVC_OP_OUTCOME, outcome, sizeof(agr_outcome), ticket); }
static int collect(agr_handle* h, agr_ticket ticket, const svc_answer& r, agr_result* out) {
    svc_host* s = h->svc;
    const bool rec = !(ticket & TICKET_OUTCOME);
    const uint64_t t = ticket & TICKET_SLOT;
    if (out) {
        memset(out, 0, sizeof *out);
        out->is_outcome = rec ? 0u : 1u;
        if (rec) {
            if ((r.w0 & 0xffu) == 0u) out->result = (int32_t)r.w1;
            else { memcpy(&out->verdict, &r.w0, 4); memcpy((uint8_t*)&out->verdict + 4, &r.w1, 4); out->rid = r.rid; svc_request_id(h, t, r.rid, out->request_id); }
        } else out->result = (int32_t)r.w0;
    }
    svc_release_run(s, t, (uint32_t)((ticket >> TICKET_RUN_SHIFT) & 15u) + 1u);
    return 0;
}
int agr_poll(agr_handle* h, agr_ticket ticket, agr_result* out) {
    if (!h || !h->svc) return fail(AGR_EINVAL, "engine was not created with AGR_CFG_COMBINE");
    svc_answer r;
    if (!svc_try(h->svc, ticket & TICKET_SLOT, &r)) return AGR_EAGAIN;
    return collect(h, ticket, r, out);
}
int agr_wait(agr_handle* h, agr_ticket ticket, agr_result* out) {
    if (!h || !h->svc) return fail(AGR_EINVAL, "engine was not created with AGR_CFG_COMBINE");
    svc_answer r;
    svc_wait(h->svc, ticket & TICKET_SLOT, &r);
    return collect(h, ticket, r, out);
}

// ------------------------------------------------------------------------------------------ K2
static int complete_locked(agr_handle* h, const agr_outcome* outs, uint32_t n, int32_t* results);

int agr_complete(agr_handle* h, const agr_outcome* outs, uint32_t n, int32_t* results) {
    if (!h || (n && !outs)) return fail(AGR_EINVAL, "NULL argument");
    if (h->svc && n >= 1 && n <= SVC_MAX_CALL) return svc_complete(h, outs, n, results);
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    return complete_locked(h, outs, n, results);
}

static int complete_locked(agr_handle* h, const agr_outcome* outs, uint32_t n, int32_t* results) {
    if (n > h->cfg.max_batch) return fail(AGR_EINVAL, "n exceeds max_batch");
    if (n == 0) return 0;
    // outcomes go to the device as they are; k2_prepare resolves the agent ids in the device agent table
    if (is_pinned(outs)) {
        CK(cudaMemcpyAsync(h->d_outs, outs, (size_t)n * sizeof(agr_outcome), cudaMemcpyHostToDevice, h->stream));
    } else {
        memcpy(h->h_outs, outs, (size_t)n * sizeof(agr_outcome));
        CK(cudaMemcpyAsync(h->d_outs, h->h_outs, (size_t)n * sizeof(agr_outcome), cudaMemcpyHostToDevice, h->stream));
    }
    sync_window(h);
    const bool timing = (h->cfg.flags & AGR_CFG_TIMING) != 0;
    if (timing) {
        for (auto& e : h->op_ev) if (!e) CK(cudaEventCreate(&e));
        CK(cudaEventRecord(h->op_ev[0], h->stream));
    }
    agr_launch_k2(h->d, h->d_outs, h->k2, n, h->stream);
    h->k2_launches += 3;
    CK(cudaGetLastError());
    if (timing) { CK(cudaEventRecord(h->op_ev[1], h->stream)); h->op_timed[0] = true; }
    CK(cudaMemcpyAsync(h->h_k2flag, h->k2.overflow, 4, cudaMemcpyDeviceToHost, h->stream));
    if (results) {
        CK(cudaMemcpyAsync(h->h_results, h->k2.results, (size_t)n * 4, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        memcpy(results, h->h_results, (size_t)n * 4);
    } else {
        CK(cudaStreamSynchronize(h->stream));
    }
    // the state transitions were applied; list entries beyond the log capacity were dropped (agr_config.log_entries)
    if (*h->h_k2flag) return fail(AGR_ENOSPC, "completed / failed log full: entries of this batch were dropped (raise agr_config.log_entries, or agr_reclaim)");
    return 0;
}

// ------------------------------------------------------------------------------------------ K3
static int ensure_out(agr_handle* h, uint32_t cap) {
    if (cap <= h->out_cap) return 0;
    uint32_t ncap = std::max<uint32_t>(cap, 1024);
    TRY(dev_regrow(h, &h->d_out_rid, ncap, false));
    TRY(dev_regrow(h, &h->d_out_slot, ncap, false));
    h->out_cap = ncap;
    return 0;
}
static int ensure_gather(agr_handle* h, size_t bytes) {
    if (bytes > h->gather_bytes) { TRY(dev_regrow(h, &h->d_gather, bytes, false)); h->gather_bytes = bytes; }
    if (bytes > h->h_gather_bytes) { TRY(host_regrow(h, &h->h_gather, bytes)); h->h_gather_bytes = bytes; }
    return 0;
}

// runs the stable partition; returns the number selected in *total (may exceed cap: then only counts are valid)
static int select_locked(agr_handle* h, int mode, uint32_t slot, const uint32_t* log, uint64_t lo, uint64_t hi,
                         uint32_t cap, uint32_t* total) {
    *total = 0;
    if (hi <= lo) return 0;
    agr_k3_params p{};
    p.mode = mode; p.slot = slot; p.log = log; p.lo = lo; p.hi = hi; p.lo_real = lo;
    if (mode != K3_LOG_AGENT) p.lo = lo & ~3ull;               // k3_mark reads the row words four rows per lane (16-byte loads)
    p.groups = (mode == K3_TICK) ? std::max<uint32_t>(1, (uint32_t)h->agent_names.size()) : 1;
    uint64_t items = hi - p.lo;
    uint64_t max_warps = std::max<uint64_t>(1, (4u << 20) / p.groups);
    uint64_t want = std::min<uint64_t>((uint64_t)h->sm_count * 128, (items + 1023) / 1024);  // several waves of 8-warp CTAs; the column scan runs over per-CTA rows
    p.nwarps = (uint32_t)std::max<uint64_t>(1, std::min(want, max_warps));
    uint64_t per = (items + p.nwarps - 1) / p.nwarps;
    per = (per + 255) & ~255ull;
    p.per_warp = (uint32_t)per;
    p.nwarps = (uint32_t)((items + per - 1) / per);
    size_t need = (size_t)p.nwarps * p.groups;
    if (need > h->matrix_entries) { TRY(dev_regrow(h, &h->d_matrix, need, false)); h->matrix_entries = need; }
    const size_t need_cta = (size_t)((p.nwarps + 7) / 8) * p.groups;
    if (need_cta > h->cta_matrix_entries) { TRY(dev_regrow(h, &h->d_cta_matrix, need_cta, false)); h->cta_matrix_entries = need_cta; }
    p.cta_matrix = h->d_cta_matrix;
    const size_t mask_words = (size_t)p.nwarps * (p.per_warp >> 5);
    if (mask_words > h->selmask_words) { TRY(dev_regrow(h, &h->d_selmask, mask_words, false)); h->selmask_words = mask_words; }
    p.selmask = h->d_selmask;
    TRY(ensure_out(h, cap));
    p.matrix = h->d_matrix; p.gtotal = h->d_gtotal; p.goff = h->d_goff;
    p.out_rid = h->d_out_rid; p.out_slot = h->d_out_slot; p.cap = cap;
    p.min_inq = (mode == K3_TICK) ? h->d_min_inq : nullptr;
    if (mode == K3_TICK) CK(cudaMemsetAsync(h->d_min_inq, 0xff, 4, h->stream));
    const bool timing = (h->cfg.flags & AGR_CFG_TIMING) != 0;
    if (timing) {
        for (auto& e : h->op_ev) if (!e) CK(cudaEventCreate(&e));
        CK(cudaEventRecord(h->op_ev[2], h->stream));
    }
    agr_launch_k3_select(h->d, p, h->sm_count, h->stream);
    h->k3_launches += 4;
    CK(cudaGetLastError());
    if (timing) { CK(cudaEventRecord(h->op_ev[3], h->stream)); h->op_timed[1] = true; }
    CK(cudaMemcpyAsync(h->h_small, h->d_goff + p.groups, 4, cudaMemcpyDeviceToHost, h->stream));
    if (mode == K3_TICK) CK(cudaMemcpyAsync(h->h_small + 1, h->d_min_inq, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    *total = h->h_small[0];
    if (mode == K3_TICK) {
        uint32_t m = h->h_small[1];
        h->scan_lo = (m == AGR_RID_NONE) ? hi : std::max<uint64_t>(h->scan_lo, p.lo + m);
    }
    return 0;
}

int agr_replay_scan(agr_handle* h, agr_dispatch* out, agr_record* recs, uint32_t cap, uint32_t* n) {
    if (!h || !n) return fail(AGR_EINVAL, "NULL argument");
    if ((h->cfg.flags & AGR_CFG_VARLEN) && recs) return fail(AGR_EINVAL, "variable-length engine: use agr_replay_scan_var to gather records");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    *n = 0;
    h->replay_scans++;
    uint32_t total = 0;
    TRY(select_locked(h, K3_TICK, 0, nullptr, h->scan_lo, ingested_bound(h), cap, &total));
    *n = total;
    if (total > cap) return fail(AGR_ECAP, "dispatch array too small");
    h->replay_dispatched += total;
    if (total == 0 || !out) return 0;
    size_t bytes = (size_t)total * 32 + (recs ? (size_t)total * AGR_REC : 0);
    TRY(ensure_gather(h, bytes));
    uint8_t* d_disp = h->d_gather;
    uint8_t* d_recs = recs ? h->d_gather + (size_t)total * 32 : nullptr;
    agr_launch_k3_gather(h->d, h->d_out_rid, nullptr, total, d_recs, d_disp, nullptr, h->stream);
    h->k3_launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->h_gather, h->d_gather, bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    memcpy(out, h->h_gather, (size_t)total * 32);
    if (recs) memcpy(recs, h->h_gather + (size_t)total * 32, (size_t)total * AGR_REC);
    return 0;
}

int agr_pending(agr_handle* h, const char* agent_id, agr_record* out, uint32_t cap, uint32_t* n) {
    if (!h || !agent_id || !n) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    *n = 0;
    int slot = agent_find(h, agent_id);
    if (slot < 0) return 0;     // LRANGE on a missing key is an empty list
    uint32_t total = 0;
    TRY(select_locked(h, K3_AGENT_PENDING, (uint32_t)slot, nullptr, h->scan_lo, ingested_bound(h), cap, &total));
    *n = total;
    if (total > cap) return fail(AGR_ECAP, "output array too small");
    if (total == 0 || !out) return 0;
    size_t bytes = (size_t)total * AGR_REC;
    TRY(ensure_gather(h, bytes));
    agr_launch_k3_gather(h->d, h->d_out_rid, nullptr, total, h->d_gather, nullptr, nullptr, h->stream);
    h->k3_launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->h_gather, h->d_gather, bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    memcpy(out, h->h_gather, bytes);
    return 0;
}

int agr_list(agr_handle* h, const char* agent_id, int which, uint8_t (*ids)[16], uint32_t cap, uint32_t* n) {
    if (!h || !agent_id || !n) return fail(AGR_EINVAL, "NULL argument");
    if (which < AGR_LIST_PENDING || which > AGR_LIST_FAILED) return fail(AGR_EINVAL, "bad list selector");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    *n = 0;
    int slot = agent_find(h, agent_id);
    if (slot < 0) return 0;
    uint32_t total = 0;
    if (which == AGR_LIST_PENDING) {
        // LRANGE: ids of expired records are still in the list; they lie below the scan's low-water mark
        TRY(select_locked(h, K3_AGENT_PENDING_IDS, (uint32_t)slot, nullptr, h->expired_total ? h->tail : h->scan_lo, ingested_bound(h), cap, &total));
    } else {
        unsigned long long lens[2];
        CK(cudaMemcpyAsync(lens, h->d.log_len, sizeof lens, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        const uint32_t* log = (which == AGR_LIST_COMPLETED) ? h->d.completed_log : h->d.failed_log;
        uint64_t len = (which == AGR_LIST_COMPLETED) ? lens[0] : lens[1];
        TRY(select_locked(h, K3_LOG_AGENT, (uint32_t)slot, log, 0, len, cap, &total));
    }
    *n = total;
    if (total > cap) return fail(AGR_ECAP, "output array too small");
    if (total == 0 || !ids) return 0;
    size_t bytes = (size_t)total * 16;
    TRY(ensure_gather(h, bytes));
    agr_launch_k3_gather(h->d, h->d_out_rid, nullptr, total, nullptr, nullptr, h->d_gather, h->stream);
    h->k3_launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->h_gather, h->d_gather, bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    memcpy(ids, h->h_gather, bytes);
    return 0;
}

// storage.Get("agent:{a}:requests:{r}") (server.go:661-662): read-only resolve in the dedupe index, then a 1-row gather
int agr_get_record(agr_handle* h, const char* agent_id, const uint8_t request_id[16], agr_record* out) {
    if (!h || !agent_id || !request_id || !out) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    int slot = agent_find(h, agent_id);
    if (slot < 0) return fail(AGR_ENOTFOUND, "request not found");
    agr_dop& op = h->h_ops[0];
    memcpy(&op.id_lo, request_id, 8); memcpy(&op.id_hi, request_id + 8, 8);
    op.slot = (uint32_t)slot; op.http = 0; op.kind = 0; op.pad = 0; op.seq = 0;
    CK(cudaMemcpyAsync(h->d_ops, h->h_ops, sizeof(agr_dop), cudaMemcpyHostToDevice, h->stream));
    sync_window(h);
    agr_launch_resolve(h->d, h->d_ops, h->d_hrid, 1, h->stream);
    h->k3_launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->h_small, h->d_hrid, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (h->h_small[0] == AGR_RID_NONE) return fail(AGR_ENOTFOUND, "request not found");
    TRY(ensure_gather(h, AGR_REC));
    agr_launch_k3_gather(h->d, h->d_hrid, nullptr, 1, h->d_gather, nullptr, nullptr, h->stream);
    h->k3_launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->h_gather, h->d_gather, AGR_REC, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    memcpy(out, h->h_gather, AGR_REC);
    return 0;
}

// ------------------------------------------------------------------------------------------ variable-length records
// rows and byte-slab space for n records of `bytes` stored bytes in all (agr_ingest_var, and the dispatcher of the single-request
// front end for a batch): *base = physical byte offset of the first.  Byte ring: the records never wrap either.  Nothing is
// reserved unless both fit.
static int reserve_var_locked(agr_handle* h, uint32_t n, uint64_t bytes, uint64_t* first, uint64_t* base) {
    uint64_t vpad = 0;
    if (!is_ring(h)) {
        if (h->vused + bytes > h->vcap) return fail(AGR_ENOSPC, "byte slab full");
    } else {
        if (bytes > h->vcap / 2) return fail(AGR_EINVAL, "batch larger than half the byte slab");
        const uint64_t at = h->vused % h->vcap;
        vpad = (at + bytes > h->vcap) ? h->vcap - at : 0;
        if (h->vused + vpad + bytes - h->vtail > h->vcap) return fail(AGR_ENOSPC, "byte slab full: agr_expire + agr_reclaim release bytes at the tail");
    }
    TRY(reserve_rows_locked(h, n, first));
    h->vused += vpad;
    *base = is_ring(h) ? h->vused % h->vcap : h->vused;
    h->vused += bytes;
    return 0;
}
int agr_ingest_var(agr_handle* h, const uint8_t* blob, const uint32_t* offsets, uint32_t n, agr_verdict* out, uint8_t (*ids)[16],
                   uint64_t* first_rid) {
    if (!h || (n && (!blob || !offsets))) return fail(AGR_EINVAL, "NULL argument");
    if (!(h->cfg.flags & AGR_CFG_VARLEN)) return fail(AGR_EINVAL, "engine was not created with AGR_CFG_VARLEN");
    auto shape_ok = [&]() -> int {
        if (offsets[0] != 0) return fail(AGR_EINVAL, "offsets[0] must be 0");
        for (uint32_t i = 0; i < n; ++i)                          // host-side shape check (lengths are part of the wire format)
            if (offsets[i + 1] < offsets[i] || !var_len_ok(offsets[i + 1] - offsets[i]))
                return fail(AGR_EINVAL, "record " + std::to_string(i) + ": length must be a multiple of 16 in [96, 8192]");
        return 0;
    };
    if (h->svc && n >= 1 && n <= SVC_MAX_CALL) { TRY(shape_ok()); return svc_ingest_var(h, blob, offsets, n, out, ids, first_rid); }
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    if (n > h->cfg.max_batch) return fail(AGR_EINVAL, "n exceeds max_batch");
    uint64_t first = 0;
    if (n == 0) { if (first_rid) *first_rid = h->rows_used; return 0; }
    const uint64_t bytes = offsets[n];
    TRY(shape_ok());
    uint64_t base = 0;
    TRY(reserve_var_locked(h, n, bytes, &first, &base));
    if (first_rid) *first_rid = first;
    cudaStream_t st = h->stream;
    CK(cudaMemcpyAsync(h->d.slab + base, blob, bytes, cudaMemcpyHostToDevice, st));
    if (is_pinned(offsets)) CK(cudaMemcpyAsync(h->d_voffsets, offsets, ((size_t)n + 1) * 4, cudaMemcpyHostToDevice, st));
    else { memcpy(h->h_voffsets, offsets, ((size_t)n + 1) * 4); CK(cudaMemcpyAsync(h->d_voffsets, h->h_voffsets, ((size_t)n + 1) * 4, cudaMemcpyHostToDevice, st)); }
    sync_window(h);
    flip_batch_words(h);
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (h->cfg.flags & AGR_CFG_TIMING) {
        if (h->tev.empty()) { h->tev.resize(2 * AGR_TIMING_RING); for (auto& e : h->tev) CK(cudaEventCreate(&e)); }
        const uint64_t k = h->tev_next++ % AGR_TIMING_RING;
        e0 = h->tev[2 * k]; e1 = h->tev[2 * k + 1];
        CK(cudaEventRecord(e0, st));
    }
    CK(agr_launch_k1_var(h->d, h->d.slab + base, h->d_voffsets, n, bytes, h->d_tile_first, (uint32_t)phys_row(h, first), base, h->sm_count, st, h->cfg.k1_variant));
    if (e1) CK(cudaEventRecord(e1, st));
    agr_launch_k1_post(h->d, (uint32_t)phys_row(h, first), n, h->sm_count, st, out ? h->d_verdicts : nullptr, ids ? h->d_ids : nullptr);
    h->k1_launches += 3;
    CK(cudaGetLastError());
    if (out) CK(cudaMemcpyAsync(h->h_verdicts, h->d_verdicts, (size_t)n * sizeof(agr_verdict), cudaMemcpyDeviceToHost, st));
    if (ids) CK(cudaMemcpyAsync(h->h_ids, h->d_ids, (size_t)n * 16, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (out) memcpy(out, h->h_verdicts, (size_t)n * sizeof(agr_verdict));
    if (ids) memcpy(ids, h->h_ids, (size_t)n * 16);
    return 0;
}

// packs the variable-length records of rows d_out_rid[0..total) into the caller's blob
static int gather_var_locked(agr_handle* h, uint32_t total, uint8_t* blob, uint64_t blob_cap, uint64_t* offsets, uint64_t* blob_bytes) {
    if (total > h->lens_cap) {
        uint32_t ncap = std::max<uint32_t>(total, 1024);
        TRY(dev_regrow(h, &h->d_lens, ncap, false));
        TRY(dev_regrow(h, &h->d_goffs, (size_t)ncap + 1, false));
        h->lens_cap = ncap;
    }
    agr_launch_var_lens(h->d, h->d_out_rid, total, h->d_lens, h->stream);
    std::vector<uint32_t> lens(total);
    CK(cudaMemcpyAsync(lens.data(), h->d_lens, (size_t)total * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    std::vector<unsigned long long> offs((size_t)total + 1);
    offs[0] = 0;
    for (uint32_t j = 0; j < total; ++j) offs[j + 1] = offs[j] + lens[j];
    *blob_bytes = offs[total];
    if (offsets) for (uint32_t j = 0; j <= total; ++j) offsets[j] = offs[j];
    if (!blob) return 0;
    if (offs[total] > blob_cap) return fail(AGR_ECAP, "blob too small");
    TRY(ensure_gather(h, (size_t)offs[total] + 16));
    CK(cudaMemcpyAsync(h->d_goffs, offs.data(), ((size_t)total + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    agr_launch_var_copy(h->d, h->d_out_rid, total, h->d_goffs, h->d_gather, h->stream);
    h->k3_launches += 2;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->h_gather, h->d_gather, (size_t)offs[total], cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    memcpy(blob, h->h_gather, (size_t)offs[total]);
    return 0;
}

int agr_replay_scan_var(agr_handle* h, agr_dispatch* out, uint8_t* blob, uint64_t blob_cap, uint64_t* offsets, uint32_t cap,
                        uint32_t* n, uint64_t* blob_bytes) {
    if (!h || !n || !blob_bytes) return fail(AGR_EINVAL, "NULL argument");
    if (!(h->cfg.flags & AGR_CFG_VARLEN)) return fail(AGR_EINVAL, "engine was not created with AGR_CFG_VARLEN");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    *n = 0; *blob_bytes = 0;
    h->replay_scans++;
    uint32_t total = 0;
    TRY(select_locked(h, K3_TICK, 0, nullptr, h->scan_lo, ingested_bound(h), cap, &total));
    *n = total;
    if (total > cap) return fail(AGR_ECAP, "dispatch array too small");
    h->replay_dispatched += total;
    if (total == 0) return 0;
    if (out) {
        TRY(ensure_gather(h, (size_t)total * 32));
        agr_launch_k3_gather(h->d, h->d_out_rid, nullptr, total, nullptr, h->d_gather, nullptr, h->stream);
        h->k3_launches += 1;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(h->h_gather, h->d_gather, (size_t)total * 32, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        memcpy(out, h->h_gather, (size_t)total * 32);
    }
    return gather_var_locked(h, total, blob, blob_cap, offsets, blob_bytes);
}

int agr_get_record_var(agr_handle* h, const char* agent_id, const uint8_t request_id[16], uint8_t* out, uint32_t cap, uint32_t* len) {
    if (!h || !agent_id || !request_id || !len) return fail(AGR_EINVAL, "NULL argument");
    if (!(h->cfg.flags & AGR_CFG_VARLEN)) return fail(AGR_EINVAL, "engine was not created with AGR_CFG_VARLEN");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    int slot = agent_find(h, agent_id);
    if (slot < 0) return fail(AGR_ENOTFOUND, "request not found");
    agr_dop& op = h->h_ops[0];
    memcpy(&op.id_lo, request_id, 8); memcpy(&op.id_hi, request_id + 8, 8);
    op.slot = (uint32_t)slot; op.http = 0; op.kind = 0; op.pad = 0; op.seq = 0;
    CK(cudaMemcpyAsync(h->d_ops, h->h_ops, sizeof(agr_dop), cudaMemcpyHostToDevice, h->stream));
    sync_window(h);
    agr_launch_resolve(h->d, h->d_ops, h->d_hrid, 1, h->stream);
    CK(cudaMemcpyAsync(h->h_small, h->d_hrid, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (h->h_small[0] == AGR_RID_NONE) return fail(AGR_ENOTFOUND, "request not found");
    TRY(ensure_out(h, 1));
    CK(cudaMemcpyAsync(h->d_out_rid, h->d_hrid, 4, cudaMemcpyDeviceToDevice, h->stream));
    uint64_t bytes = 0;
    std::vector<uint8_t> tmp(AGR_VAR_MAX_RECORD);
    uint64_t offs[2];
    TRY(gather_var_locked(h, 1, tmp.data(), tmp.size(), offs, &bytes));
    *len = (uint32_t)bytes;
    if (bytes > cap || !out) return out ? fail(AGR_ECAP, "output buffer too small") : 0;
    memcpy(out, tmp.data(), bytes);
    return 0;
}

// ------------------------------------------------------------------------------------------ stored responses
static int resolve_one_locked(agr_handle* h, const char* agent_id, const uint8_t request_id[16], uint32_t* rid) {
    int slot = agent_find(h, agent_id);
    if (slot < 0) return fail(AGR_ENOTFOUND, "request not found");
    agr_dop& op = h->h_ops[0];
    memcpy(&op.id_lo, request_id, 8); memcpy(&op.id_hi, request_id + 8, 8);
    op.slot = (uint32_t)slot; op.http = 0; op.kind = 0; op.pad = 0; op.seq = 0;
    CK(cudaMemcpyAsync(h->d_ops, h->h_ops, sizeof(agr_dop), cudaMemcpyHostToDevice, h->stream));
    sync_window(h);
    agr_launch_resolve(h->d, h->d_ops, h->d_hrid, 1, h->stream);
    h->k3_launches += 1;
    CK(cudaMemcpyAsync(h->h_small, h->d_hrid, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (h->h_small[0] == AGR_RID_NONE) return fail(AGR_ENOTFOUND, "request not found");
    *rid = h->h_small[0];
    return 0;
}

// which: 0 = response (hdr_len leading bytes are its flattened headers), 1 = error text
static int store_bytes_locked(agr_handle* h, const char* agent_id, const uint8_t request_id[16], int which, const uint8_t* a, uint32_t alen,
                              const uint8_t* b, uint32_t blen) {
    uint32_t rid = 0;
    TRY(resolve_one_locked(h, agent_id, request_id, &rid));
    const uint32_t len = alen + blen;
    const uint64_t need = ((uint64_t)len + 15u) & ~15ull;
    unsigned long long off;
    if (!is_ring(h)) {
        if (h->resp_used + len > h->resp_cap) return fail(AGR_ENOSPC, "response slab full");
        off = h->resp_used;
        h->resp_used += need;
    } else {                                                     // byte ring: a blob never wraps; agr_reclaim advances resp_tail
        if (need > h->resp_cap / 2) return fail(AGR_ENOSPC, "response larger than half the response slab");
        const uint64_t at = h->resp_used % h->resp_cap;
        const uint64_t pad = (at + need > h->resp_cap) ? h->resp_cap - at : 0;
        if (h->resp_used + pad + need - h->resp_tail > h->resp_cap)
            return fail(AGR_ENOSPC, "response slab full: agr_reclaim releases the bytes of released rows");
        h->resp_used += pad;
        off = h->resp_used % h->resp_cap;                        // the rows keep PHYSICAL offsets
        h->resp_used += need;
    }
    if (alen) CK(cudaMemcpyAsync(h->d_resp + off, a, alen, cudaMemcpyHostToDevice, h->stream));
    if (blen) CK(cudaMemcpyAsync(h->d_resp + off + alen, b, blen, cudaMemcpyHostToDevice, h->stream));
    if (which == 0) {
        CK(cudaMemcpyAsync(h->d_resp_off + rid, &off, 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->d_resp_len + rid, &len, 4, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->d_resp_hlen + rid, &alen, 4, cudaMemcpyHostToDevice, h->stream));
    } else {
        CK(cudaMemcpyAsync(h->d_err_off + rid, &off, 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->d_err_len + rid, &len, 4, cudaMemcpyHostToDevice, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}
int agr_store_response(agr_handle* h, const char* agent_id, const uint8_t request_id[16], const uint8_t* headers, uint32_t hdr_len,
                       const uint8_t* body, uint32_t body_len) {
    if (!h || !agent_id || !request_id || (hdr_len && !headers) || (body_len && !body)) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    return store_bytes_locked(h, agent_id, request_id, 0, headers, hdr_len, body, body_len);
}
int agr_store_response_body(agr_handle* h, const char* agent_id, const uint8_t request_id[16], const uint8_t* bytes, uint32_t len) {
    return agr_store_response(h, agent_id, request_id, nullptr, 0, bytes, len);
}
int agr_store_error_text(agr_handle* h, const char* agent_id, const uint8_t request_id[16], const char* text, uint32_t len) {
    if (!h || !agent_id || !request_id || (len && !text)) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    return store_bytes_locked(h, agent_id, request_id, 1, (const uint8_t*)text, len, nullptr, 0);
}

int agr_get_response_body(agr_handle* h, const char* agent_id, const uint8_t request_id[16], uint8_t* out, uint32_t cap, uint32_t* len) {
    if (!h || !agent_id || !request_id || !len) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    uint32_t rid = 0;
    TRY(resolve_one_locked(h, agent_id, request_id, &rid));
    unsigned long long off = 0; uint32_t l = 0;
    CK(cudaMemcpyAsync(&off, h->d_resp_off + rid, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(&l, h->d_resp_len + rid, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    *len = l;
    if (l > cap || !out) return (out && l > cap) ? fail(AGR_ECAP, "output buffer too small") : 0;
    if (l) { CK(cudaMemcpyAsync(out, h->d_resp + off, l, cudaMemcpyDeviceToHost, h->stream)); CK(cudaStreamSynchronize(h->stream)); }
    return 0;
}

// ------------------------------------------------------------------------------------------ K5: JSON wire form
// Encodes n records (rows d_rids[0..n) or first_rid + [0..n)) into h->d_json; *total = bytes.  Offsets stay in h->d_joff.
static int json_encode_locked(agr_handle* h, const uint32_t* d_rids, uint64_t first_rid, uint32_t n, bool array, uint64_t* total, bool roundtrip = false) {
    *total = 0;
    if (n == 0) return 0;
    if (n > h->j_cap) {
        const uint32_t cap = std::max<uint32_t>(n, 1024);
        TRY(dev_regrow(h, &h->d_jlen, cap, false));
        TRY(dev_regrow(h, &h->d_joff, (size_t)cap + 1, false));
        TRY(dev_regrow(h, &h->d_jchunk, (size_t)agr_k5_chunks(cap) + 1, false));
        h->j_cap = cap;
    }
    agr_k5_params p{};
    p.rids = d_rids; p.first_l = first_rid; p.n = n; p.array = array ? 1u : 0u; p.roundtrip = roundtrip ? 1u : 0u;
    sync_window(h);
    p.len = h->d_jlen; p.off = h->d_joff; p.chunk_sum = h->d_jchunk; p.out = nullptr;
    p.bytes = h->d_resp; p.resp_off = h->d_resp_off; p.resp_len = h->d_resp_len; p.resp_hlen = h->d_resp_hlen;
    p.err_off = h->d_err_off; p.err_len = h->d_err_len; p.ptime = h->d.ptime;
    const bool timing = (h->cfg.flags & AGR_CFG_TIMING) != 0;
    if (timing) {
        for (auto& e : h->op_ev) if (!e) CK(cudaEventCreate(&e));
        CK(cudaEventRecord(h->op_ev[4], h->stream));
    }
    agr_launch_k5_measure(h->d, p, h->stream);
    CK(cudaGetLastError());
    unsigned long long tot = 0;
    CK(cudaMemcpyAsync(&tot, h->d_jchunk + agr_k5_chunks(n), 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (tot + 16 > h->json_cap) {
        const uint64_t cap = std::max<uint64_t>(tot + tot / 4 + 16, 1 << 16);
        TRY(dev_regrow(h, &h->d_json, (size_t)cap, false));
        h->json_cap = cap;
    }
    p.out = h->d_json;
    agr_launch_k5_emit(h->d, p, h->stream);
    CK(cudaGetLastError());
    if (timing) { CK(cudaEventRecord(h->op_ev[5], h->stream)); h->op_timed[2] = true; }
    h->k5_launches += 3;
    *total = tot;
    return 0;
}
static int json_copy_out(agr_handle* h, uint64_t total, uint8_t* out, uint64_t cap, uint64_t* len) {
    *len = total;
    if (!out) { CK(cudaStreamSynchronize(h->stream)); return 0; }
    if (total > cap) return fail(AGR_ECAP, "output buffer too small");
    if (total) CK(cudaMemcpyAsync(out, h->d_json, (size_t)total, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int agr_rows_json(agr_handle* h, uint64_t first_rid, uint32_t n, int as_array, uint8_t* out, uint64_t cap, uint64_t* len, uint64_t* offsets) {
    if (!h || !len) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    if (first_rid + n > h->rows_used || first_rid < h->tail) return fail(AGR_EINVAL, "row range outside the rows in use");
    uint64_t total = 0;
    TRY(json_encode_locked(h, nullptr, first_rid, n, (as_array & 1) != 0, &total, (as_array & 2) != 0));
    if (n == 0 && (as_array & 1)) {                              // json.Marshal of a nil slice
        *len = 4;
        if (out) { if (cap < 4) return fail(AGR_ECAP, "output buffer too small"); memcpy(out, "null", 4); }
        if (offsets) offsets[0] = 0;
        return 0;
    }
    if (offsets && n) CK(cudaMemcpyAsync(offsets, h->d_joff, ((size_t)n + 1) * 8, cudaMemcpyDeviceToHost, h->stream));
    else if (offsets) offsets[0] = 0;
    return json_copy_out(h, total, out, cap, len);
}

int agr_pending_json(agr_handle* h, const char* agent_id, uint8_t* out, uint64_t cap, uint64_t* len, uint32_t* count) {
    if (!h || !agent_id || !len) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    if (count) *count = 0;
    uint32_t total_rows = 0;
    int slot = agent_find(h, agent_id);
    if (slot >= 0) {
        const uint32_t cap0 = std::max<uint32_t>(h->out_cap, 1024);
        TRY(select_locked(h, K3_AGENT_PENDING, (uint32_t)slot, nullptr, h->scan_lo, ingested_bound(h), cap0, &total_rows));
        if (total_rows > cap0)                                   // counts only: run again with room for all of it
            TRY(select_locked(h, K3_AGENT_PENDING, (uint32_t)slot, nullptr, h->scan_lo, ingested_bound(h), total_rows, &total_rows));
    }
    if (count) *count = total_rows;
    if (total_rows == 0) {                                       // var requests []*Request stays nil (requests.go:204): "null"
        *len = 4;
        if (out) { if (cap < 4) return fail(AGR_ECAP, "output buffer too small"); memcpy(out, "null", 4); }
        return 0;
    }
    uint64_t total = 0;
    TRY(json_encode_locked(h, h->d_out_rid, 0, total_rows, true, &total, true));   // GetPendingRequests unmarshals every record
    return json_copy_out(h, total, out, cap, len);
}

int agr_get_record_json(agr_handle* h, const char* agent_id, const uint8_t request_id[16], uint8_t* out, uint32_t cap, uint32_t* len) {
    if (!h || !agent_id || !request_id || !len) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    uint32_t rid = 0;
    TRY(resolve_one_locked(h, agent_id, request_id, &rid));
    uint64_t total = 0, l = 0;
    TRY(json_encode_locked(h, h->d_hrid, 0, 1, false, &total));   // k2.hrid[0] = the physical row resolve_one_locked found
    int rc = json_copy_out(h, total, out, cap, &l);
    *len = (uint32_t)l;
    return rc;
}

// ------------------------------------------------------------------------------------------ durability
struct snap_header {
    char magic[8];                 // "AGRSNAP3"
    uint32_t flags, n_agents, shard, gen;
    uint64_t rows_used, vused, log_len[2], id_secret, scan_lo, resp_used, expired_total, tail, released_total, slab_rows, vtail, vcap, resp_tail, resp_cap;
};
static int dump_dev(agr_handle* h, FILE* f, const void* dsrc, size_t bytes) {
    const size_t chunk = h->bounce_bytes;
    for (size_t o = 0; o < bytes; o += chunk) {
        const size_t m = std::min(chunk, bytes - o);
        CK(cudaMemcpyAsync(h->bounce[0], (const uint8_t*)dsrc + o, m, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (fwrite(h->bounce[0], 1, m, f) != m) return fail(AGR_EINVAL, "snapshot: short write");
    }
    return 0;
}
static int load_dev(agr_handle* h, FILE* f, void* ddst, size_t bytes) {
    const size_t chunk = h->bounce_bytes;
    for (size_t o = 0; o < bytes; o += chunk) {
        const size_t m = std::min(chunk, bytes - o);
        if (fread(h->bounce[0], 1, m, f) != m) return fail(AGR_EINVAL, "restore: short read");
        CK(cudaMemcpyAsync((uint8_t*)ddst + o, h->bounce[0], m, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    return 0;
}

int agr_snapshot(agr_handle* h, const char* path) {
    if (!h || !path) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    FILE* f = fopen(path, "wb");
    if (!f) return fail(AGR_EINVAL, std::string("snapshot: cannot open ") + path);
    snap_header hd{};
    memcpy(hd.magic, "AGRSNAP3", 8);
    hd.flags = h->cfg.flags & (AGR_CFG_PERSISTENCE | AGR_CFG_MINT_IDS | AGR_CFG_VARLEN | AGR_CFG_RING);
    hd.n_agents = (uint32_t)h->agent_names.size(); hd.shard = h->d.shard_id; hd.gen = h->d.id_gen;
    hd.rows_used = h->rows_used; hd.vused = h->vused; hd.id_secret = h->d.id_secret; hd.scan_lo = h->scan_lo;
    hd.resp_used = h->resp_used; hd.expired_total = h->expired_total; hd.tail = h->tail; hd.released_total = h->released_total; hd.slab_rows = h->cfg.slab_rows; hd.vtail = h->vtail; hd.vcap = h->vcap; hd.resp_tail = h->resp_tail; hd.resp_cap = h->resp_cap;
    unsigned long long lens[2];
    int rc = 0;
    auto done = [&](int r) { fclose(f); return r; };
    if (cudaMemcpy(lens, h->d.log_len, sizeof lens, cudaMemcpyDeviceToHost) != cudaSuccess) return done(fail(AGR_ECUDA, "snapshot: log_len"));
    hd.log_len[0] = lens[0]; hd.log_len[1] = lens[1];
    if (fwrite(&hd, sizeof hd, 1, f) != 1) return done(fail(AGR_EINVAL, "snapshot: short write"));
    for (uint32_t a = 0; a < hd.n_agents; ++a) {
        char name[AGR_AGENT_ID_BYTES] = {0};
        strncpy(name, h->agent_names[a].c_str(), AGR_AGENT_ID_BYTES - 1);
        fwrite(name, 1, AGR_AGENT_ID_BYTES, f); fwrite(&h->agent_status[a], 1, 1, f);
    }
    const size_t R = (size_t)rows_span(h);
    const size_t slab_bytes = (h->cfg.flags & AGR_CFG_VARLEN) ? (size_t)(is_ring(h) ? std::min<uint64_t>(hd.vused, h->vcap) : hd.vused) : R * AGR_REC;
    if ((rc = dump_dev(h, f, h->d.slab, slab_bytes)) < 0) return done(rc);
    if ((rc = dump_dev(h, f, h->d.state, R * 4)) < 0) return done(rc);
    if ((rc = dump_dev(h, f, h->d.route, R * 4)) < 0) return done(rc);
    if ((rc = dump_dev(h, f, h->d.aux, R * 4)) < 0) return done(rc);
    if ((rc = dump_dev(h, f, h->d.cksum, R * 8)) < 0) return done(rc);
    if (h->cfg.flags & AGR_CFG_VARLEN) {
        if ((rc = dump_dev(h, f, h->d.voff, R * 8)) < 0) return done(rc);
        if ((rc = dump_dev(h, f, h->d.vlen, R * 4)) < 0) return done(rc);
    }
    if ((rc = dump_dev(h, f, h->d.completed_log, (size_t)lens[0] * 4)) < 0) return done(rc);
    if ((rc = dump_dev(h, f, h->d.failed_log, (size_t)lens[1] * 4)) < 0) return done(rc);
    if ((rc = dump_dev(h, f, h->d_resp, (size_t)(is_ring(h) ? std::min<uint64_t>(hd.resp_used, h->resp_cap) : hd.resp_used))) < 0) return done(rc);
    if ((rc = dump_dev(h, f, h->d_resp_off, R * 8)) < 0) return done(rc);
    if ((rc = dump_dev(h, f, h->d_resp_len, R * 4)) < 0) return done(rc);
    if ((rc = dump_dev(h, f, h->d_resp_hlen, R * 4)) < 0) return done(rc);
    if ((rc = dump_dev(h, f, h->d_err_off, R * 8)) < 0) return done(rc);
    if ((rc = dump_dev(h, f, h->d_err_len, R * 4)) < 0) return done(rc);
    if ((rc = dump_dev(h, f, h->d.ptime, R * 8)) < 0) return done(rc);
    if ((rc = dump_dev(h, f, h->d.mtime, R * 8)) < 0) return done(rc);
    return done(0);
}

int agr_restore(const agr_config* cfg, const char* path, agr_handle** out) {
    if (!cfg || !path || !out) return fail(AGR_EINVAL, "NULL argument");
    *out = nullptr;
    FILE* f = fopen(path, "rb");
    if (!f) return fail(AGR_EINVAL, std::string("restore: cannot open ") + path);
    snap_header hd{};
    if (fread(&hd, sizeof hd, 1, f) != 1 || memcmp(hd.magic, "AGRSNAP3", 8) != 0) { fclose(f); return fail(AGR_EINVAL, "restore: not a snapshot"); }
    agr_config c = *cfg;
    if (c.flags == 0) c.flags = AGR_CFG_PERSISTENCE;
    const uint32_t mode_bits = AGR_CFG_MINT_IDS | AGR_CFG_VARLEN | AGR_CFG_RING;
    if ((c.flags & mode_bits) != (hd.flags & mode_bits)) { fclose(f); return fail(AGR_EINVAL, "restore: id mode / record form differ from the snapshot"); }
    if (c.id_secret == 0) c.id_secret = hd.id_secret;
    if (c.id_secret != hd.id_secret) { fclose(f); return fail(AGR_EINVAL, "restore: id_secret differs from the snapshot"); }
    agr_handle* h = nullptr;
    int rc = agr_create(&c, &h);
    if (rc < 0) { fclose(f); return rc; }
    auto bail = [&](int r) { std::string keep = g_err; fclose(f); agr_destroy(h); g_err = keep; return r; };
    const bool snap_ring = (hd.flags & AGR_CFG_RING) != 0;
    if (!snap_ring && hd.resp_used > h->resp_cap) return bail(fail(AGR_ENOSPC, "restore: stored responses larger than resp_bytes"));
    if (snap_ring && hd.resp_cap != h->resp_cap) return bail(fail(AGR_EINVAL, "restore: a ring snapshot needs the same resp_bytes"));
    if (snap_ring && (hd.flags & AGR_CFG_VARLEN) && hd.vcap != h->vcap) return bail(fail(AGR_EINVAL, "restore: a ring snapshot needs the same vslab_bytes"));
    if (snap_ring && hd.slab_rows != h->cfg.slab_rows) return bail(fail(AGR_EINVAL, "restore: a ring snapshot needs the same slab_rows (rows live at logical mod slab_rows)"));
    if ((!snap_ring && hd.rows_used > h->cfg.slab_rows) || hd.log_len[0] > h->d.log_cap || hd.log_len[1] > h->d.log_cap || ((hd.flags & AGR_CFG_VARLEN) && !snap_ring && hd.vused > h->vcap))
        return bail(fail(AGR_ENOSPC, "restore: snapshot larger than the configured capacities"));
    for (uint32_t a = 0; a < hd.n_agents; ++a) {
        char name[AGR_AGENT_ID_BYTES]; uint8_t st;
        if (fread(name, 1, AGR_AGENT_ID_BYTES, f) != AGR_AGENT_ID_BYTES || fread(&st, 1, 1, f) != 1) return bail(fail(AGR_EINVAL, "restore: short read"));
        name[AGR_AGENT_ID_BYTES - 1] = 0;
        const bool removed = (st == AG_STATUS_REMOVED);
        if ((rc = agr_set_agent_state(h, name, removed ? (uint8_t)AGR_AGENT_STOPPED : st)) < 0) return bail(rc);
        if (removed) { HLock lk(h); h->agent_status[a] = AG_STATUS_REMOVED; if ((rc = push_agent_status(h, a, AG_STATUS_REMOVED)) < 0) return bail(rc); }
    }
    HLock lk(h);
    const size_t R = snap_ring ? (size_t)std::min<uint64_t>(hd.rows_used, hd.slab_rows) : (size_t)hd.rows_used;
    const size_t slab_bytes = (hd.flags & AGR_CFG_VARLEN) ? (size_t)(snap_ring ? std::min<uint64_t>(hd.vused, hd.vcap) : hd.vused) : R * AGR_REC;
    if ((rc = load_dev(h, f, h->d.slab, slab_bytes)) < 0) return bail(rc);
    if ((rc = load_dev(h, f, h->d.state, R * 4)) < 0) return bail(rc);
    if ((rc = load_dev(h, f, h->d.route, R * 4)) < 0) return bail(rc);
    if ((rc = load_dev(h, f, h->d.aux, R * 4)) < 0) return bail(rc);
    if ((rc = load_dev(h, f, h->d.cksum, R * 8)) < 0) return bail(rc);
    if (hd.flags & AGR_CFG_VARLEN) {
        if ((rc = load_dev(h, f, h->d.voff, R * 8)) < 0) return bail(rc);
        if ((rc = load_dev(h, f, h->d.vlen, R * 4)) < 0) return bail(rc);
    }
    if ((rc = load_dev(h, f, h->d.completed_log, (size_t)hd.log_len[0] * 4)) < 0) return bail(rc);
    if ((rc = load_dev(h, f, h->d.failed_log, (size_t)hd.log_len[1] * 4)) < 0) return bail(rc);
    if ((rc = load_dev(h, f, h->d_resp, (size_t)(snap_ring ? std::min<uint64_t>(hd.resp_used, hd.resp_cap) : hd.resp_used))) < 0) return bail(rc);
    if ((rc = load_dev(h, f, h->d_resp_off, R * 8)) < 0) return bail(rc);
    if ((rc = load_dev(h, f, h->d_resp_len, R * 4)) < 0) return bail(rc);
    if ((rc = load_dev(h, f, h->d_resp_hlen, R * 4)) < 0) return bail(rc);
    if ((rc = load_dev(h, f, h->d_err_off, R * 8)) < 0) return bail(rc);
    if ((rc = load_dev(h, f, h->d_err_len, R * 4)) < 0) return bail(rc);
    if ((rc = load_dev(h, f, h->d.ptime, R * 8)) < 0) return bail(rc);
    if ((rc = load_dev(h, f, h->d.mtime, R * 8)) < 0) return bail(rc);
    h->resp_used = hd.resp_used; h->resp_tail = hd.resp_tail; h->expired_total = hd.expired_total;
    unsigned long long lens[2] = {hd.log_len[0], hd.log_len[1]};
    if (cudaMemcpy(h->d.log_len, lens, sizeof lens, cudaMemcpyHostToDevice) != cudaSuccess) return bail(fail(AGR_ECUDA, "restore: log_len"));
    h->rows_used = hd.rows_used; h->vused = hd.vused; h->vtail = hd.vtail; h->scan_lo = hd.scan_lo;
    h->d.shard_id = hd.shard; h->d.id_gen = hd.gen; h->tail = hd.tail; h->released_total = hd.released_total; sync_window(h);
    h->d.idx_base = h->tail;
    cudaMemsetAsync(h->d.cmin, 0, (size_t)(h->cfg.slab_rows / AGR_CHUNK_ROWS + 2) * 8, h->stream);       // time bounds unknown: the first sweep recomputes them
    if (!(hd.flags & AGR_CFG_MINT_IDS) && R) {        // hash-id mode: rebuild the dedupe index from the restored rows
        agr_launch_reindex(h->d, (uint32_t)R, h->stream);
        h->k1_launches += 1;
        if (cudaStreamSynchronize(h->stream) != cudaSuccess) return bail(fail(AGR_ECUDA, "restore: reindex"));
    }
    fclose(f);
    *out = h;
    return 0;
}

int agr_expire(agr_handle* h, uint64_t now, uint64_t ttl, uint64_t* expired) {
    if (!h) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    unsigned long long* d_cnt = expired ? (unsigned long long*)(h->d.ctr + C_NCTR - 1) : nullptr;     // last counter slot as scratch
    if (d_cnt) CK(cudaMemsetAsync(d_cnt, 0, 8, h->stream));
    sync_window(h);
    if ((!is_ring(h) || (h->cfg.flags & AGR_CFG_VARLEN)) && h->rows_used > h->sweep_clean) {
        // append-only slabs and variable-length engines: K1 does not keep the chunks' time bounds (k1_note_time); the chunks that
        // received rows since the last sweep are marked "unknown" here and get their exact bound back from this sweep
        const uint64_t R = h->cfg.slab_rows, lo = std::max(h->sweep_clean, h->tail), hi = h->rows_used;
        if (is_ring(h) && hi - lo >= R) CK(cudaMemsetAsync(h->d.cmin, 0, (size_t)(R / AGR_CHUNK_ROWS + 1) * 8, h->stream));
        else if (hi > lo) {
            const uint64_t p0 = phys_row(h, lo), p1 = phys_row(h, hi - 1);
            auto zero = [&](uint64_t a, uint64_t b) { return cudaMemsetAsync(h->d.cmin + a / AGR_CHUNK_ROWS, 0, (size_t)(b / AGR_CHUNK_ROWS - a / AGR_CHUNK_ROWS + 1) * 8, h->stream); };
            if (p0 <= p1) CK(zero(p0, p1)); else { CK(zero(p0, R - 1)); CK(zero(0, p1)); }
        }
        h->sweep_clean = ingested_bound(h);
    }
    agr_launch_expire(h->d, rows_span(h), now, ttl, d_cnt, h->stream);
    h->k3_launches += 1;
    CK(cudaGetLastError());
    if (!expired) {                       // no count wanted: stay asynchronous (the sweep is stream-ordered before whatever follows)
        h->expired_total = std::max<uint64_t>(h->expired_total, 1);   // "records may have expired": the list views widen their scan
        return 0;
    }
    unsigned long long v = 0;
    CK(cudaMemcpyAsync(&v, d_cnt, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->expired_total += v;
    *expired = v;
    return 0;
}

// what one scan of the ring's tail reports back (device -> pinned host, one 32-byte copy)
struct reclaim_result { uint32_t off, pad; unsigned long long lens[2]; unsigned long long voff; };

// enqueues the scan: first stored row behind the tail (k_first_live), the log lengths and — variable-length mode — the byte
// offset of that row's record, packed by the scan's last CTA straight into pinned memory; nothing waits here
static int reclaim_scan_launch(agr_handle* h, uint64_t bound) {
    sync_window(h);
    // (the scan's two scratch words re-arm themselves, and its last CTA writes the result into the pinned buffer: one launch)
    agr_launch_first_live(h->d, bound - h->tail, is_ring(h) && !(h->cfg.flags & AGR_CFG_VARLEN), h->d_reclaim_scratch, h->h_reclaim, h->stream);
    CK(cudaGetLastError());
    if (!h->reclaim_ev) CK(cudaEventCreateWithFlags(&h->reclaim_ev, cudaEventDisableTiming));
    CK(cudaEventRecord(h->reclaim_ev, h->stream));
    h->reclaim_bound = bound;
    h->reclaim_pending = true;
    h->k3_launches += 2;
    return 0;
}

// releases what a finished scan found: rows [tail, tail + count) go back to the ring
static int reclaim_apply(agr_handle* h, uint64_t* released) {
    h->reclaim_pending = false;
    const reclaim_result r = *reinterpret_cast<const reclaim_result*>(h->h_reclaim);
    const uint64_t bound = h->reclaim_bound;
    const uint64_t count = (r.off == 0xffffffffu) ? bound - h->tail : r.off;
    if (count == 0) return 0;
    sync_window(h);
    agr_launch_release_rows(h->d, (uint32_t)count, h->d_resp_len, h->d_resp_hlen, h->d_err_len, h->stream);
    h->k3_launches += 1;
    for (int k = 0; k < 2; ++k) {                                              // completed, failed
        if (!r.lens[k]) continue;
        uint32_t*& log = k == 0 ? h->d.completed_log : h->d.failed_log;
        agr_launch_log_compact(h->d, log, r.lens[k], (uint32_t)count, h->d_log_scratch, h->d_lc_chunks, h->d.log_len + k, h->stream);
        CK(cudaGetLastError());
        std::swap(log, h->d_log_scratch);                                      // the compacted copy becomes the log
        h->k3_launches += 3;
    }
    h->tail += count;
    h->released_total += count;
    if (h->scan_lo < h->tail) h->scan_lo = h->tail;
    sync_window(h);
    if (!(h->cfg.flags & AGR_CFG_MINT_IDS)) {
        // hash-id mode: the released rows' ids must leave the dedupe index before their rows are reused.  Open addressing
        // has no cheap delete; a release is a periodic event, so the index is rebuilt from the live window instead.
        CK(cudaMemsetAsync(h->d.table, 0, (size_t)(h->d.table_mask + 1) * sizeof(agr_slot), h->stream));
        h->d.idx_base = h->tail;                                              // row words of the rebuilt index are relative to the new tail
        const uint64_t R = h->cfg.slab_rows, live = h->rows_used - h->tail, p0 = h->tail % R;
        const uint64_t n0 = std::min<uint64_t>(live, R - p0);
        agr_launch_reindex_range(h->d, (uint32_t)p0, (uint32_t)n0, h->stream);
        if (live > n0) agr_launch_reindex_range(h->d, 0, (uint32_t)(live - n0), h->stream);
        CK(cudaGetLastError());
        h->k1_launches += 2;
    }
    if (h->resp_used != h->resp_tail) {   // the response / error byte ring: its tail follows the oldest blob a live row still refers to
        unsigned long long* d_span = (unsigned long long*)(h->d.ctr + C_NCTR - 1);              // last counter slot as scratch
        CK(cudaMemsetAsync(d_span, 0, 8, h->stream));
        agr_launch_bytes_span(h->d, h->resp_used % h->resp_cap, h->resp_cap, h->d_resp_off, h->d_resp_len, h->d_err_off, h->d_err_len, d_span, h->stream);
        CK(cudaGetLastError());
        unsigned long long span = 0;
        CK(cudaMemcpyAsync(&span, d_span, 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        h->resp_tail = h->resp_used - span;
        h->k3_launches += 1;
    }
    if (h->cfg.flags & AGR_CFG_VARLEN) {                          // the byte ring's tail follows: first byte of the first live record
        if (r.off == 0xffffffffu) h->vtail = (bound == h->rows_used) ? h->vused : h->vtail;
        else {
            uint64_t used = (h->vused % h->vcap + h->vcap - r.voff) % h->vcap;
            if (used == 0) used = h->vcap;                         // head == tail with live records: the ring is exactly full
            h->vtail = h->vused - used;
        }
    }
    if (released) *released = count;
    return 0;
}

// AGR_CFG_RING: hand the rows at the tail that hold no record any more (expired or never stored) back to the ring, up to
// the first row that still does, and drop their entries from the completed / failed logs.
int agr_reclaim(agr_handle* h, uint64_t* released) {
    if (!h) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    if (released) *released = 0;
    if (!is_ring(h)) return fail(AGR_EINVAL, "engine was not created with AGR_CFG_RING");
    uint64_t got = 0;
    if (h->reclaim_pending) { CK(cudaEventSynchronize(h->reclaim_ev)); TRY(reclaim_apply(h, &got)); }   // a scan agr_reclaim_async left behind
    const uint64_t bound = ingested_bound(h);                                  // reserved rows that K1 has not filled yet are not "dead"
    if (bound > h->tail) {
        TRY(reclaim_scan_launch(h, bound));
        CK(cudaStreamSynchronize(h->stream));                                  // the only host round trip
        uint64_t more = 0;
        TRY(reclaim_apply(h, &more));
        got += more;
    }
    if (released) *released = got;
    return 0;
}
// The same without the host round trip in the caller's way: releases what the scan started by the PREVIOUS call found (it has
// long finished) and starts the next scan.  A ring that is maintained every step lags one step behind and never waits.
int agr_reclaim_async(agr_handle* h, uint64_t* released) {
    if (!h) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    if (released) *released = 0;
    if (!is_ring(h)) return fail(AGR_EINVAL, "engine was not created with AGR_CFG_RING");
    if (h->reclaim_pending) { CK(cudaEventSynchronize(h->reclaim_ev)); TRY(reclaim_apply(h, released)); }
    const uint64_t bound = ingested_bound(h);
    if (bound > h->tail) TRY(reclaim_scan_launch(h, bound));
    return 0;
}

int agr_verify(agr_handle* h, uint64_t* rows_checked, uint64_t* bad) {
    if (!h || !bad) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    unsigned long long* d_bad = (unsigned long long*)(h->d.ctr + C_NCTR - 1);     // last counter slot as scratch
    CK(cudaMemsetAsync(d_bad, 0, 8, h->stream));
    sync_window(h);
    agr_launch_verify(h->d, rows_span(h), d_bad, h->stream);
    h->k3_launches += 1;
    CK(cudaGetLastError());
    unsigned long long v = 0;
    CK(cudaMemcpyAsync(&v, d_bad, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    *bad = v;
    if (rows_checked) *rows_checked = rows_span(h);
    return 0;
}

// ------------------------------------------------------------------------------------------ stats
int agr_stats_get(agr_handle* h, agr_stats* out) {
    if (!h || !out) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    unsigned long long c[C_NCTR], lens[2];
    CK(cudaMemcpyAsync(c, h->d.ctr, sizeof c, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(lens, h->d.log_len, sizeof lens, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    memset(out, 0, sizeof *out);
    out->rows_used = h->rows_used; out->rows_cap = h->cfg.slab_rows;
    out->ingested = c[C_INGESTED]; out->stored = c[C_STORED]; out->replay_flagged = c[C_REPLAY];
    out->dedupe_hits = c[C_DEDUPE_HITS]; out->forwarded = c[C_FORWARDED]; out->queued = c[C_QUEUED];
    out->unavailable = c[C_UNAVAILABLE]; out->not_found = c[C_NOT_FOUND]; out->dup_ids = c[C_DUP_IDS];
    out->completions = c[C_COMPLETIONS]; out->completion_misses = c[C_COMPLETION_MISSES];
    out->failures = c[C_FAILURES]; out->dead_lettered = c[C_DEAD_LETTERED]; out->dial_errors = c[C_DIAL_ERRORS];
    out->replay_scans = h->replay_scans; out->replay_dispatched = h->replay_dispatched;
    out->completed_log_len = lens[0]; out->failed_log_len = lens[1];
    out->k1_launches = h->k1_launches; out->k2_launches = h->k2_launches;
    out->k3_launches = h->k3_launches; out->k4_launches = h->k4_launches; out->k5_launches = h->k5_launches; out->rows_tail = h->tail;
    out->malformed = c[C_BAD_LEN]; out->log_overflow = c[C_LOG_OVERFLOW];
    if (h->svc) { out->svc_batches = h->svc->batches.load(); out->svc_ops = h->svc->ops.load(); }
    out->agents = (uint32_t)h->agent_names.size(); out->device = (uint32_t)h->device;
    return 0;
}

// ------------------------------------------------------------------------------------------ K4 exchange
static int nccl_load() {
    if (g_nccl.lib) return 0;
    void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) return fail(AGR_ECOMM, std::string("dlopen libnccl.so.2: ") + dlerror());
#define SYM(field, name) *(void**)(&g_nccl.field) = dlsym(lib, name); if (!g_nccl.field) return fail(AGR_ECOMM, "libnccl.so.2 lacks " name)
    SYM(GetUniqueId, "ncclGetUniqueId"); SYM(CommInitRank, "ncclCommInitRank"); SYM(CommDestroy, "ncclCommDestroy");
    SYM(Send, "ncclSend"); SYM(Recv, "ncclRecv"); SYM(GroupStart, "ncclGroupStart"); SYM(GroupEnd, "ncclGroupEnd");
    SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
    g_nccl.lib = lib;
    return 0;
}
#define NK(call) do { ncclResult_t r_ = (call); if (r_ != ncclSuccess) return fail(AGR_ECOMM, std::string(#call) + ": " + g_nccl.GetErrorString(r_)); } while (0)

int agr_comm_unique_id(uint8_t out[128]) {
    if (!out) return fail(AGR_EINVAL, "NULL argument");
    TRY(nccl_load());
    ncclUniqueId id;
    NK(g_nccl.GetUniqueId(&id));
    memcpy(out, id.internal, 128);
    return 0;
}

int agr_comm_init(agr_handle* h, const uint8_t id[128], int rank, int world) {
    if (!h || !id) return fail(AGR_EINVAL, "NULL argument");
    if (world < 1 || world > 32 || rank < 0 || rank >= world) return fail(AGR_EINVAL, "bad rank / world (1..32 shards)");
    TRY(nccl_load());
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    ncclUniqueId uid; memcpy(uid.internal, id, 128);
    NK(g_nccl.CommInitRank(&h->comm, world, uid, rank));
    h->rank = rank; h->world = world;
    h->d.shard_id = (uint32_t)rank;
    const size_t mb = h->cfg.max_batch;
    TRY(dev_alloc(h, &h->d_stage, mb * sizeof(agr_outcome), false));   // outcomes before binning (records are binned in their slab rows)
    TRY(dev_alloc(h, &h->d_send, mb * AGR_REC, false));
    TRY(dev_alloc(h, &h->d_owner, mb, false));
    TRY(dev_alloc(h, &h->d_perm, mb, false));
    h->k4_nwarps = (uint32_t)std::min<size_t>((size_t)h->sm_count * 32, std::max<size_t>(1, (mb + 1023) / 1024));
    TRY(dev_alloc(h, &h->d_k4matrix, (size_t)h->k4_nwarps * 32, false));
    TRY(dev_alloc(h, &h->d_k4cnt, (size_t)4 * 40, true));
    TRY(dev_alloc(h, &h->d_xverd, 2 * mb, false));
    TRY(dev_alloc(h, &h->d_vback, mb, false));
    TRY(dev_alloc(h, &h->d_vout, mb, false));
    // K2 over local + received outcomes: scratch for 2 * max_batch ops
    TRY(dev_alloc(h, &h->d_outs, 2 * mb, false));
    TRY(k2_scratch_alloc(h, 2 * mb));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// Shared first half of the exchanges: find every item's owner (K4 count + scan), swap the per-peer counts with one grouped
// send/recv, and lay out the owner-major send offsets and the source-major receive offsets.  `d_items` are the items on the
// device: the staging buffer (outcomes), or the slab rows the batch was DMA'd into (records, in-place mode).
struct exchange_plan {
    agr_k4_params p{};
    uint32_t G = 1, me = 0, scnt[32], rcnt[32], soff[33], roff[33], n_local = 0, n_recv = 0;
    uint32_t recv_res_base = 0;      // index of the first received item's result in the result array
};
static int exchange_begin(agr_handle* h, uint8_t* d_items, uint32_t item_bytes, uint32_t agent_off, uint32_t n, bool inplace, exchange_plan& x) {
    if (!h->comm) return fail(AGR_ECOMM, "agr_comm_init has not been called on this handle");
    if (n > h->cfg.max_batch) return fail(AGR_EINVAL, "n exceeds max_batch");
    x.G = (uint32_t)h->world; x.me = (uint32_t)h->rank;
    cudaStream_t st = h->stream;
    uint32_t* d_gtotal = h->d_k4cnt; uint32_t* d_goff = h->d_k4cnt + 40; uint32_t* d_rcnt = h->d_k4cnt + 80;
    agr_k4_params& p = x.p;
    p.items = d_items; p.items_rw = d_items; p.inplace = inplace ? 1u : 0u;
    p.item_bytes = item_bytes; p.agent_off = agent_off; p.n = n; p.G = x.G; p.me = x.me;
    uint32_t per = (n + h->k4_nwarps - 1) / std::max<uint32_t>(1, h->k4_nwarps);
    per = std::max<uint32_t>(32, (per + 31) & ~31u);
    p.per_warp = per; p.nwarps = std::max<uint32_t>(1, (n + per - 1) / per);
    p.matrix = h->d_k4matrix; p.gtotal = d_gtotal; p.goff = d_goff; p.owner = h->d_owner; p.perm = h->d_perm;
    agr_launch_k4_count(p, st);
    h->k4_launches += 2;
    CK(cudaGetLastError());
    NK(g_nccl.GroupStart());
    for (uint32_t q = 0; q < x.G; ++q) {
        NK(g_nccl.Send(d_gtotal + q, 1, ncclUint32, (int)q, h->comm, st));
        NK(g_nccl.Recv(d_rcnt + q, 1, ncclUint32, (int)q, h->comm, st));
    }
    NK(g_nccl.GroupEnd());
    // the one host round trip of the exchange: ncclSend / ncclRecv take their element counts from the host, and the rows for
    // the records that arrive have to be reserved
    uint32_t* hc = h->h_small;                       // [0..31] send counts, [32..63] receive counts
    CK(cudaMemcpyAsync(hc, d_gtotal, x.G * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(hc + 32, d_rcnt, x.G * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    x.soff[0] = 0; x.roff[0] = 0;
    for (uint32_t q = 0; q < x.G; ++q) {
        x.scnt[q] = hc[q]; x.rcnt[q] = (q == x.me) ? 0 : hc[32 + q];
        // in-place mode: the send buffer holds the peers' segments only
        x.soff[q + 1] = x.soff[q] + ((inplace && q == x.me) ? 0u : x.scnt[q]); x.roff[q + 1] = x.roff[q] + x.rcnt[q];
    }
    x.n_local = x.scnt[x.me]; x.n_recv = x.roff[x.G];
    x.recv_res_base = inplace ? n : x.n_local;
    if ((inplace ? n : x.n_local) + x.n_recv > 2 * h->cfg.max_batch) return fail(AGR_ENOSPC, "received more items than 2 * max_batch");
    return 0;
}
// the all-to-all itself: peer segments of `send` to their owners, landing at recv_base in source-rank order
static int exchange_payload(agr_handle* h, const exchange_plan& x, const uint8_t* send, uint8_t* recv_base, size_t item_bytes) {
    NK(g_nccl.GroupStart());
    for (uint32_t q = 0; q < x.G; ++q) {
        if (q == x.me) continue;
        if (x.scnt[q]) NK(g_nccl.Send(send + (size_t)x.soff[q] * item_bytes, (size_t)x.scnt[q] * item_bytes, ncclUint8, (int)q, h->comm, h->stream));
        if (x.rcnt[q]) NK(g_nccl.Recv(recv_base + (size_t)x.roff[q] * item_bytes, (size_t)x.rcnt[q] * item_bytes, ncclUint8, (int)q, h->comm, h->stream));
    }
    NK(g_nccl.GroupEnd());
    return 0;
}
// results of the received items back to where they came from (owner-major at the reporter), then the caller's order
static int exchange_results(agr_handle* h, const exchange_plan& x, const uint8_t* res_all /*own items first, then received*/, uint8_t* back,
                            uint8_t* out_dev, uint32_t res_bytes) {
    NK(g_nccl.GroupStart());
    for (uint32_t q = 0; q < x.G; ++q) {
        if (q == x.me) continue;
        if (x.rcnt[q]) NK(g_nccl.Send(res_all + (size_t)(x.recv_res_base + x.roff[q]) * res_bytes, (size_t)x.rcnt[q] * res_bytes, ncclUint8, (int)q, h->comm, h->stream));
        if (x.scnt[q]) NK(g_nccl.Recv(back + (size_t)x.soff[q] * res_bytes, (size_t)x.scnt[q] * res_bytes, ncclUint8, (int)q, h->comm, h->stream));
    }
    NK(g_nccl.GroupEnd());
    if (x.p.n) {
        agr_launch_k4_unpermute(x.p, res_all, back, out_dev, res_bytes, h->stream);
        h->k4_launches += 1;
        CK(cudaGetLastError());
    }
    return 0;
}
static void exchange_fill_info(const exchange_plan& x, uint32_t n, uint64_t first, uint64_t recv_first, agr_exchange_info* info) {
    if (!info) return;
    memset(info, 0, sizeof *info);
    info->world = x.G; info->rank = x.me; info->n_local = x.n_local; info->n_sent = n - x.n_local; info->n_received = x.n_recv;
    info->first_rid = first; info->recv_first_rid = recv_first;
    for (uint32_t q = 0; q < x.G; ++q) { info->sent_to[q] = (q == x.me) ? 0 : x.scnt[q]; info->received_from[q] = x.rcnt[q]; }
}

// The exchange over a batch that already lies in slab rows [first, first + n) (DMA'd there by agr_ingest_sharded, or filled on
// the device).  Records of this shard's agents never move: K4 only copies the records owned by a PEER into the send buffer and
// marks their rows empty; received records land in rows reserved behind the batch, straight from the all-to-all.
static int sharded_rows_locked(agr_handle* h, uint64_t first, uint32_t n, agr_verdict* out, agr_exchange_info* info) {
    exchange_plan x;
    uint8_t* rows = h->d.slab + phys_row(h, first) * AGR_REC;
    TRY(exchange_begin(h, rows, AGR_REC, AGR_OFF_AGENT_ID, n, true, x));
    uint64_t first2 = h->rows_used;
    if (x.n_recv) TRY(reserve_rows_locked(h, x.n_recv, &first2));
    const uint32_t n_remote = n - x.n_local;
    x.p.local_dst = nullptr; x.p.send_dst = h->d_send;
    if (n_remote) { agr_launch_k4_scatter(x.p, h->stream); h->k4_launches += 1; CK(cudaGetLastError()); }
    // K1 over the batch's own rows (rows emptied by K4 are skipped) — runs while the all-to-all below moves the peers' records
    if (n) {
        const uint32_t keep = h->d.cfg_flags;
        if (n_remote) h->d.cfg_flags |= AGR_CFGI_HOLES;
        const int rc = launch_k1_locked(h, first, n, h->d_xverd);
        h->d.cfg_flags = keep;
        TRY(rc);
    }
    // the all-to-all: every peer segment to its owner, landing directly in the owner's slab rows
    TRY(exchange_payload(h, x, h->d_send, h->d.slab + phys_row(h, first2) * AGR_REC, AGR_REC));
    // K1 at the owner over the received rows (own host's records first, then peers by rank: the merge order)
    if (x.n_recv) TRY(launch_k1_locked(h, first2, x.n_recv, h->d_xverd + n));
    // verdicts back to where the records came from, restored to the caller's order
    TRY(exchange_results(h, x, (const uint8_t*)h->d_xverd, (uint8_t*)h->d_vback, (uint8_t*)h->d_vout, sizeof(agr_verdict)));
    if (n && out) CK(cudaMemcpyAsync(h->h_verdicts, h->d_vout, (size_t)n * sizeof(agr_verdict), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (n && out) memcpy(out, h->h_verdicts, (size_t)n * sizeof(agr_verdict));
    exchange_fill_info(x, n, first, first2, info);
    return 0;
}

int agr_ingest_sharded(agr_handle* h, const agr_record* recs, uint32_t n, agr_verdict* out, agr_exchange_info* info) {
    if (!h || (n && !recs)) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    if (!h->comm) return fail(AGR_ECOMM, "agr_comm_init has not been called on this handle");
    if (n > h->cfg.max_batch) return fail(AGR_EINVAL, "n exceeds max_batch");
    uint64_t first = h->rows_used;
    if (n) {
        TRY(reserve_rows_locked(h, n, &first));
        // the batch goes STRAIGHT into its slab rows, in chunks on the copy stream (a pageable source through the bounce buffers)
        const bool src_pinned = is_pinned(recs);
        while (h->chunk_ev.size() < 2) { cudaEvent_t e; CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); h->chunk_ev.push_back(e); }
        CK(cudaEventRecord(h->chunk_ev[0], h->stream));
        CK(cudaStreamWaitEvent(h->copy_stream, h->chunk_ev[0], 0));
        uint8_t* dst = h->d.slab + phys_row(h, first) * AGR_REC;
        const size_t bytes = (size_t)n * AGR_REC;
        if (src_pinned) CK(cudaMemcpyAsync(dst, recs, bytes, cudaMemcpyHostToDevice, h->copy_stream));
        else {
            int bk = 0;
            for (size_t o = 0; o < bytes;) {
                const size_t piece = std::min(h->bounce_bytes, bytes - o);
                CK(cudaEventSynchronize(h->bounce_ev[bk]));
                par_memcpy(h->bounce[bk], (const uint8_t*)recs + o, piece);
                CK(cudaMemcpyAsync(dst + o, h->bounce[bk], piece, cudaMemcpyHostToDevice, h->copy_stream));
                CK(cudaEventRecord(h->bounce_ev[bk], h->copy_stream));
                o += piece; bk ^= 1;
            }
        }
        CK(cudaEventRecord(h->chunk_ev[1], h->copy_stream));
        CK(cudaStreamWaitEvent(h->stream, h->chunk_ev[1], 0));
    }
    return sharded_rows_locked(h, first, n, out, info);
}
// The same over rows the caller reserved (agr_reserve_rows) and filled on the device: the exchange with the batch resident in HBM.
int agr_ingest_sharded_rows(agr_handle* h, uint64_t first_rid, uint32_t n, agr_verdict* out, agr_exchange_info* info) {
    if (!h) return fail(AGR_EINVAL, "NULL handle");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    if (!h->comm) return fail(AGR_ECOMM, "agr_comm_init has not been called on this handle");
    if (first_rid + n > h->rows_used) return fail(AGR_EINVAL, "rows not reserved");
    if (n > h->cfg.max_batch) return fail(AGR_EINVAL, "n exceeds max_batch");
    if (!h->resv.empty()) resv_remove(h, first_rid, first_rid + n);
    return sharded_rows_locked(h, first_rid, n, out, info);
}

int agr_complete_sharded(agr_handle* h, const agr_outcome* outs, uint32_t n, int32_t* results, agr_exchange_info* info) {
    if (!h || (n && !outs)) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    exchange_plan x;
    if (!h->comm) return fail(AGR_ECOMM, "agr_comm_init has not been called on this handle");
    if (n > h->cfg.max_batch) return fail(AGR_EINVAL, "n exceeds max_batch");
    if (n) CK(cudaMemcpyAsync(h->d_stage, outs, (size_t)n * sizeof(agr_outcome), cudaMemcpyHostToDevice, h->stream));
    TRY(exchange_begin(h, h->d_stage, sizeof(agr_outcome), 16, n, false, x));
    const uint32_t total = x.n_local + x.n_recv;
    // pack: own outcomes straight into the K2 input array, peer segments into the send buffer
    x.p.local_dst = (uint8_t*)h->d_outs; x.p.send_dst = h->d_send;
    if (n) { agr_launch_k4_scatter(x.p, h->stream); h->k4_launches += 1; CK(cudaGetLastError()); }
    TRY(exchange_payload(h, x, h->d_send, (uint8_t*)(h->d_outs + x.n_local), sizeof(agr_outcome)));
    // K2 at the owner over local + received outcomes (own host first, then peers by rank)
    if (total) {
        sync_window(h);
        agr_launch_k2(h->d, h->d_outs, h->k2, total, h->stream);
        h->k2_launches += 3;
        CK(cudaGetLastError());
    }
    TRY(exchange_results(h, x, (const uint8_t*)h->k2.results, (uint8_t*)h->d_vback, (uint8_t*)h->d_vout, 4));
    if (n && results) CK(cudaMemcpyAsync(h->h_results, h->d_vout, (size_t)n * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (n && results) memcpy(results, h->h_results, (size_t)n * 4);
    exchange_fill_info(x, n, 0, 0, info);
    return 0;
}

int agr_debug_read(agr_handle* h, int which, uint64_t first_rid, uint32_t n, void* out) {
    if (!h || (n && !out)) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    if (!is_ring(h) && first_rid + n > h->cfg.slab_rows) return fail(AGR_EINVAL, "row range out of bounds");
    if (is_ring(h) && (first_rid + n > h->rows_used || n > h->cfg.slab_rows)) return fail(AGR_EINVAL, "row range out of bounds");
    const uint8_t* base = nullptr; size_t w = 4;
    switch (which) {
        case AGR_DBG_STATE: base = (const uint8_t*)h->d.state; break;
        case AGR_DBG_ROUTE: base = (const uint8_t*)h->d.route; break;
        case AGR_DBG_AUX: base = (const uint8_t*)h->d.aux; break;
        case AGR_DBG_CKSUM: base = (const uint8_t*)h->d.cksum; w = 8; break;
        default: return fail(AGR_EINVAL, "bad array selector");
    }
    const uint64_t p0 = phys_row(h, first_rid);
    const uint64_t n0 = is_ring(h) ? std::min<uint64_t>(n, h->cfg.slab_rows - p0) : n;          // a logical range may wrap once
    if (n0) CK(cudaMemcpyAsync(out, base + p0 * w, (size_t)n0 * w, cudaMemcpyDeviceToHost, h->stream));
    if (n > n0) CK(cudaMemcpyAsync((uint8_t*)out + n0 * w, base, (size_t)(n - n0) * w, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int agr_op_time(agr_handle* h, int which, double* ms) {
    if (!h || !ms || which < 0 || which > 2) return fail(AGR_EINVAL, "bad argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    if (!h->op_timed[which]) return fail(AGR_ENOTFOUND, "no timed launch of that group yet (needs AGR_CFG_TIMING)");
    CK(cudaStreamSynchronize(h->stream));
    float f = 0;
    CK(cudaEventElapsedTime(&f, h->op_ev[2 * which], h->op_ev[2 * which + 1]));
    *ms = f;
    return 0;
}

int agr_kernel_time(agr_handle* h, double* sum_ms, uint64_t* launches) {
    if (!h || !sum_ms || !launches) return fail(AGR_EINVAL, "NULL argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    *sum_ms = 0; *launches = 0;
    uint64_t from = h->tev_read;
    if (h->tev_next - from > AGR_TIMING_RING) from = h->tev_next - AGR_TIMING_RING;
    for (uint64_t i = from; i < h->tev_next; ++i) {
        float ms = 0;
        const uint64_t k = i % AGR_TIMING_RING;
        CK(cudaEventElapsedTime(&ms, h->tev[2 * k], h->tev[2 * k + 1]));
        *sum_ms += ms; (*launches)++;
    }
    h->tev_read = h->tev_next;
    h->timing_calls = 0;                       // the next launch is a timed one again (stride, k1_variant bits 16..23)
    return 0;
}

// ------------------------------------------------------------------------------------------ synthetic stream
int agr_synth_bind_mint(agr_handle* h, agr_synth* s, uint64_t base_rid) {
    if (!h || !s) return fail(AGR_EINVAL, "NULL argument");
    if (!(h->cfg.flags & AGR_CFG_MINT_IDS)) return fail(AGR_EINVAL, "engine was not created with AGR_CFG_MINT_IDS");
    s->mint = 1; s->mint_base_rid = base_rid; s->mint_secret = h->d.id_secret; s->mint_shard = h->d.shard_id; s->mint_gen = h->d.id_gen;
    return 0;
}

static agr_synth_dev synth_params(const agr_synth* s, const unsigned long long* cdf) {
    agr_synth_dev p;
    p.mint = s->mint; p.mint_shard = s->mint_shard; p.mint_gen = s->mint_gen; p.pad = 0;
    p.mint_base_rid = s->mint_base_rid; p.mint_secret = s->mint_secret;
    p.seed = s->seed; p.n_agents = s->n_agents; p.dup_permille = s->dup_permille;
    p.agent_nanos0 = s->agent_nanos0 ? s->agent_nanos0 : 1700000000000000000ULL;
    p.cdf = cdf;
    return p;
}
// Zipf(s = zipf_milli / 1000) cumulative thresholds in pure integer arithmetic, so the table (and therefore the
// stream) is bit-identical on every host: weight_k = 2^40 * 2^-(s * log2(k+1)), log2 in 32.32 fixed point by
// repeated squaring, 2^-f as a product of the constants 2^-(2^-(b+1)) obtained from an integer square-root chain.
typedef unsigned __int128 u128_t;
static unsigned long long fx_log2(unsigned long long x) {        // integer x >= 1 -> log2(x) in 32.32
    unsigned long long ip = 0;
    for (unsigned long long v = x; v >= 2; v >>= 1) ip++;
    u128_t m = (u128_t)x << (63 - ip);                           // mantissa in [1,2) as Q1.63
    unsigned long long frac = 0;
    for (int b = 31; b >= 0; --b) {
        m = (m * m) >> 63;                                       // square: value in [1,4)
        if (m >> 64) { m >>= 1; frac |= (1ULL << b); }           // >= 2: emit a one bit, renormalise
    }
    return (ip << 32) | frac;
}
static unsigned long long isqrt128(u128_t v) {
    u128_t lo = 0, hi = (u128_t)1 << 64;
    while (lo + 1 < hi) { u128_t mid = (lo + hi) >> 1; if (mid * mid <= v) lo = mid; else hi = mid; }
    return (unsigned long long)lo;
}
static void zipf_cdf(uint32_t n, uint32_t zipf_milli, std::vector<unsigned long long>& cdf) {
    unsigned long long r[32];                                    // r[b] = 2^-(2^-(b+1)) in Q0.64
    r[0] = isqrt128((u128_t)1 << 127);
    for (int k = 1; k < 32; ++k) r[k] = isqrt128((u128_t)r[k - 1] << 64);
    std::vector<unsigned long long> w(n);
    u128_t total = 0;
    for (uint32_t k = 0; k < n; ++k) {
        const unsigned long long y = (unsigned long long)(((u128_t)fx_log2((unsigned long long)k + 1) * zipf_milli) / 1000);
        const unsigned long long ip = y >> 32, fr = y & 0xffffffffULL;
        u128_t a = (u128_t)1 << 64;                              // 1.0 in Q1.64
        for (int b = 0; b < 32; ++b)
            if (fr & (1ULL << (31 - b))) a = (a * r[b]) >> 64;
        unsigned long long wk = ip >= 40 ? 0 : (unsigned long long)(a >> 24) >> ip;   // 2^40 * 2^-y
        w[k] = wk ? wk : 1;
        total += w[k];
    }
    cdf.resize(n);
    u128_t run = 0;
    for (uint32_t k = 0; k < n; ++k) {
        run += w[k];
        u128_t t = (run << 64) / total;
        cdf[k] = (k + 1 == n || (t >> 64)) ? ~0ULL : (unsigned long long)t;
    }
}

int agr_synth_agent_id(const agr_synth* s, uint32_t k, char out[AGR_AGENT_ID_BYTES]) {
    if (!s || !out) return fail(AGR_EINVAL, "NULL argument");
    unsigned long long n0 = s->agent_nanos0 ? s->agent_nanos0 : 1700000000000000000ULL;
    agr_synth_agent_name(n0 + (unsigned long long)k * 1000003ULL, out);
    return 0;
}
int agr_synth_fill_host(const agr_synth* s, uint64_t first_index, uint32_t n, agr_record* out) {
    if (!s || (n && !out) || s->n_agents == 0) return fail(AGR_EINVAL, "bad argument");
    std::vector<unsigned long long> cdf;
    if (s->zipf_milli) zipf_cdf(s->n_agents, s->zipf_milli, cdf);
    agr_synth_dev p = synth_params(s, s->zipf_milli ? cdf.data() : nullptr);
    for (uint32_t i = 0; i < n; ++i) agr_synth_record(p, first_index + i, (unsigned char*)&out[i]);
    return 0;
}
int agr_synth_fill_rows(agr_handle* h, const agr_synth* s, uint64_t first_index, uint64_t first_rid, uint32_t n) {
    if (!h || !s || s->n_agents == 0) return fail(AGR_EINVAL, "bad argument");
    HLock lk(h);
    CK(cudaSetDevice(h->device));
    if (first_rid + n > h->rows_used) return fail(AGR_EINVAL, "rows not reserved");
    const unsigned long long* dcdf = nullptr;
    if (s->zipf_milli) {
        std::vector<unsigned long long> cdf;
        zipf_cdf(s->n_agents, s->zipf_milli, cdf);
        if (h->cdf_n < s->n_agents) { TRY(dev_regrow(h, &h->d_cdf, s->n_agents, false)); h->cdf_n = s->n_agents; }
        CK(cudaMemcpyAsync(h->d_cdf, cdf.data(), (size_t)s->n_agents * 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        dcdf = h->d_cdf;
    }
    agr_launch_synth(h->d.slab + phys_row(h, first_rid) * AGR_REC, synth_params(s, dcdf), first_index, n, h->stream);
    CK(cudaGetLastError());                                      // (stream-ordered before whatever reads the rows: no wait here)
    return 0;
}

uint64_t agr_agent_hash(const char* agent_id) { return agent_id ? agr_fnv1a64(agent_id, AGR_AGENT_ID_BYTES) : 0; }
uint32_t agr_agent_shard(const char* agent_id, uint32_t n_shards) {
    return n_shards ? (uint32_t)(agr_agent_hash(agent_id) % n_shards) : 0;
}

}  // extern "C"
