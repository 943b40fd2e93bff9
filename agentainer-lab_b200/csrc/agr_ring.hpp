// agr_ring.hpp — the CALLERS' side of the single-request ring (AGR_CFG_COMBINE; layout and protocol: agr_svc.h).
//
// Everything a calling thread does to hand one operation over and to collect its answer, as templates over the host-side ring
// object H (agr_engine.cu's svc_host; tests/ring_sim.cpp's stand-in).  H provides:
//   svc_res* res; uint8_t* payload; std::atomic<uint32_t>* ready;          pinned, device-mapped in the engine
//   std::atomic<uint64_t> head, scanned; std::atomic<uint32_t> waiters; uint32_t spin_cpus;
//   std::atomic<bool> sleeping; std::mutex smu; std::condition_variable scv;   the dispatcher's sleep / wake-up
//   uint32_t* lens;                                                        runs only (svc_submit_run, svc_scan_run): pinned, device-mapped
// The dispatcher (engine) or its stand-in (simulation) consumes ready words in slot order, keeps `scanned` = first slot whose
// ready word it has not consumed, and sees to it that every consumed operation other than SVC_OP_SKIP gets its 16-byte answer.
#pragma once
#include <stdint.h>
#include <string.h>
#include <atomic>
#include <condition_variable>
#include <mutex>
#include <immintrin.h>
#include <sched.h>
#include <time.h>
#include <sys/prctl.h>
#include "agr_svc.h"

// The answer cells are written by the GPU (one 16-byte PCIe store) and by host threads (svc_release, svc_fail_ops); their tag word
// is the synchronising one.  Acquire / release accesses through the compiler's atomic builtins: plain MOVs on x86-64, and a form
// ThreadSanitizer understands when this header runs against the CPU stand-in (tests/ring_sim.cpp).
static inline uint32_t svc_tag_word(const svc_res* r) { return __atomic_load_n(&r->w[3], __ATOMIC_ACQUIRE); }
static inline uint32_t svc_word(const svc_res* r, int k) { return __atomic_load_n(&r->w[k], __ATOMIC_RELAXED); }

static inline void cpu_relax(uint32_t& spins) {
    if (++spins < 4096u) _mm_pause();
    else { sched_yield(); }
}

// Slot reuse.  A caller that draws slot number a (lap = a / SVC_SLOTS of the ring) may overwrite the slot's payload and ready
// word only when the op one lap earlier is completely over: the dispatcher has consumed its ready word, the GPU has answered it
// and its caller has collected the answer (svc_release puts SVC_COLLECTED into the answer's tag).  The first two depend on
// the dispatcher and the GPU alone and are waited for.  The third depends on ANOTHER CALLER — the holder of that ticket, who may
// itself be inside a submit, waiting for one of our uncollected tickets — so it is never waited for beyond a short spin:
// the slot is published as a no-op instead (the ring moves on, the uncollected answer stays intact) and the caller is told to
// collect and come again (AGR_EAGAIN from agr_submit_*; the blocking calls, which hold no tickets, simply take the next slot).
template <class H>
static bool svc_slot_free(H* s, uint64_t a, uint32_t slot, uint32_t lap) {
    if (!lap) return true;
    const uint32_t prev = svc_tag(a - SVC_SLOTS);
    // usual case: the previous lap's op was a real one and is over (its tag in the cell says all three at once — and the ready
    // word, which sits in the dispatcher's cache, need not be read)
    if ((svc_tag_word(&s->res[slot]) >> 16) == (prev | SVC_COLLECTED)) return true;
    uint32_t w = 0;
    while (s->scanned.load(std::memory_order_acquire) <= a - SVC_SLOTS) cpu_relax(w);     // its ready word has been consumed
    const uint32_t rw = s->ready[slot].load(std::memory_order_acquire);
    if ((rw & 3u) != SVC_OP_SKIP) {
        w = 0;
        while (((svc_tag_word(&s->res[slot]) >> 16) & 0x7fffu) != prev) cpu_relax(w);                // answered (GPU, or svc_fail_ops)
    }
    // the previous lap was a no-op: the cell holds an older answer (or none at all)
    for (uint32_t k = 0; k < 2000u; ++k) {                                                   // ~0.1 ms of patience
        const uint32_t t = svc_tag_word(&s->res[slot]) >> 16;
        if (t == 0u || (t & SVC_COLLECTED)) return true;
        _mm_pause();
    }
    return false;
}
// hands ONE operation over.  true: *abs is its slot (ticket); false: the slot it drew was not free (see above).
template <class H>
static bool svc_submit_one(H* s, uint32_t kind, const void* item, size_t item_bytes, uint64_t* abs) {
    const uint64_t a = s->head.fetch_add(1, std::memory_order_relaxed);
    const uint32_t slot = (uint32_t)(a & (SVC_SLOTS - 1u)), lap = (uint32_t)(a / SVC_SLOTS);
    const bool ok = svc_slot_free(s, a, slot, lap);
    if (ok) {
        // streaming stores: the slot's lines were last written by another core a lap ago and are read next by the GPU (DMA),
        // so pulling them into this core's cache first (read-for-ownership) would only cost a miss per line
        __m128i* dst = reinterpret_cast<__m128i*>(s->payload + (size_t)slot * SVC_PAYLOAD);
        const __m128i* src = reinterpret_cast<const __m128i*>(item);
        for (size_t k = 0; k < item_bytes / 16; ++k) _mm_stream_si128(dst + k, _mm_loadu_si128(src + k));
        _mm_sfence();
    }
    s->ready[slot].store(((lap + 1u) << 2) | (ok ? kind : (uint32_t)SVC_OP_SKIP), std::memory_order_release);
    if (s->sleeping.load(std::memory_order_seq_cst)) { std::lock_guard<std::mutex> lk(s->smu); s->scv.notify_one(); }
    *abs = a;
    return ok;
}

// ---- runs (AGR_CFG_VARLEN): a record of stored length len takes svc_run_slots(len) consecutive slots, possibly across the ring's
// end.  Every slot of the run obeys the slot-reuse rule above, the GPU answers every cell of it (the continuation cells with
// their tag only, before the head's answer) and the collector releases every cell, so svc_slot_free needs nothing new.
static inline uint32_t svc_run_slots(uint32_t len) { return (len + SVC_PAYLOAD - 1u) / SVC_PAYLOAD; }
// hands ONE variable-length record over.  true: *abs is its head slot (ticket); false: some slot of the run was not free, and
// the whole run has been published as no-ops.
template <class H>
static bool svc_submit_run(H* s, const uint8_t* rec, uint32_t len, uint64_t* abs) {
    const uint32_t k = svc_run_slots(len);
    const uint64_t a = s->head.fetch_add(k, std::memory_order_relaxed);
    bool ok = true;
    for (uint32_t j = 0; j < k && ok; ++j) {
        const uint64_t b = a + j;
        ok = svc_slot_free(s, b, (uint32_t)(b & (SVC_SLOTS - 1u)), (uint32_t)(b / SVC_SLOTS));
    }
    if (ok) {
        for (uint32_t j = 0; j < k; ++j) {                       // slot by slot: the run may cross the ring's end
            __m128i* dst = reinterpret_cast<__m128i*>(s->payload + (size_t)((a + j) & (SVC_SLOTS - 1u)) * SVC_PAYLOAD);
            const __m128i* src = reinterpret_cast<const __m128i*>(rec + (size_t)j * SVC_PAYLOAD);
            const uint32_t n = (j + 1u == k ? len - j * SVC_PAYLOAD : SVC_PAYLOAD) / 16u;
            for (uint32_t c = 0; c < n; ++c) _mm_stream_si128(dst + c, _mm_loadu_si128(src + c));
        }
        _mm_sfence();
        __atomic_store_n(&s->lens[a & (SVC_SLOTS - 1u)], len, __ATOMIC_RELAXED);
        for (uint32_t j = 1; j < k; ++j) {
            const uint64_t b = a + j;
            s->ready[b & (SVC_SLOTS - 1u)].store(((uint32_t)(b / SVC_SLOTS) + 1u) << 2 | SVC_OP_CONT, std::memory_order_relaxed);
        }
        // the head last: a scanner that sees it published sees the length word and the whole run
        s->ready[a & (SVC_SLOTS - 1u)].store(((uint32_t)(a / SVC_SLOTS) + 1u) << 2 | SVC_OP_RECORD, std::memory_order_release);
    } else {
        // a slot's ready word may be overwritten only once the dispatcher has consumed the previous lap's (the slots after the one
        // that failed were not looked at)
        uint32_t w = 0;
        while (s->scanned.load(std::memory_order_acquire) + SVC_SLOTS <= a + k - 1u) cpu_relax(w);
        for (uint32_t j = 0; j < k; ++j) {
            const uint64_t b = a + j;
            s->ready[b & (SVC_SLOTS - 1u)].store(((uint32_t)(b / SVC_SLOTS) + 1u) << 2 | SVC_OP_SKIP, std::memory_order_release);
        }
    }
    if (s->sleeping.load(std::memory_order_seq_cst)) { std::lock_guard<std::mutex> lk(s->smu); s->scv.notify_one(); }
    *abs = a;
    return ok;
}

struct svc_answer { uint32_t w0, w1; uint64_t rid; };
template <class H>
static inline bool svc_try(H* s, uint64_t a, svc_answer* out) {
    const svc_res* r = s->res + (a & (SVC_SLOTS - 1u));
    const uint32_t w3 = svc_tag_word(r);
    if ((w3 >> 16) != svc_tag(a)) return false;
    out->w0 = svc_word(r, 0); out->w1 = svc_word(r, 1); out->rid = (uint64_t)svc_word(r, 2) | ((uint64_t)(w3 & 0xffffu) << 32);
    return true;
}
// Blocking wait.  The first spin_cpus waiters spin (the answer is ~20 us away); waiters beyond that many would only burn the
// process's CPU allowance against each other (a container with a CPU quota throttles ALL its threads once it is spent), so they
// sleep in short naps instead.
template <class H>
static inline void svc_wait(H* s, uint64_t a, svc_answer* out) {
    if (svc_try(s, a, out)) return;
    const uint32_t me = s->waiters.fetch_add(1, std::memory_order_relaxed);
    if (me < s->spin_cpus) {
        uint32_t w = 0;
        while (!svc_try(s, a, out)) cpu_relax(w);
    } else {
        static thread_local bool slack_set = false;
        if (!slack_set) { prctl(PR_SET_TIMERSLACK, 1000UL, 0, 0, 0); slack_set = true; }   // naps of tens of us, not the default +50 us
        struct timespec ts = {0, 25000};
        while (!svc_try(s, a, out)) nanosleep(&ts, nullptr);
    }
    s->waiters.fetch_sub(1, std::memory_order_relaxed);
}
template <class H>
static inline void svc_release(H* s, uint64_t a) {       // everything of the answer (and of the payload) has been read
    __atomic_store_n(&s->res[a & (SVC_SLOTS - 1u)].w[3], (svc_tag(a) | SVC_COLLECTED) << 16, __ATOMIC_RELEASE);
}
template <class H>
static inline void svc_release_run(H* s, uint64_t a, uint32_t k) {      // every cell of a run (k slots from a)
    for (uint32_t j = 0; j < k; ++j) svc_release(s, a + j);
}

// ---- the dispatcher's side of the ready words
// Grows the contiguous published prefix [taken, *to) by whatever has been published since: at most SVC_MAX_OPS operations and
// max_records records per batch.  A slot is looked at until it is published and never again (re-reading the callers' ready words
// every iteration keeps pulling their cache lines away from the cores that write them), and an operation's kind is noted in
// kinds[] (2 bits each, the batch descriptor's form) AT THAT MOMENT: a no-op slot may be published again, for the next lap, as soon
// as `scanned` has passed it.  Publishes the new scan position.
template <class H>
static inline void svc_scan(H* s, const uint64_t taken, uint64_t* to, uint32_t* nrec, uint32_t* kinds, const uint32_t max_records) {
    while (*to - taken < SVC_MAX_OPS) {
        const uint32_t slot = (uint32_t)(*to & (SVC_SLOTS - 1u));
        const uint32_t rw = s->ready[slot].load(std::memory_order_acquire);
        if ((rw >> 2) != (uint32_t)(*to / SVC_SLOTS) + 1u) break;
        if ((rw & 3u) == SVC_OP_RECORD) { if (*nrec == max_records) break; (*nrec)++; }
        kinds[(*to - taken) >> 4] |= (rw & 3u) << (((*to - taken) & 15u) * 2u);
        (*to)++;
    }
    if (*to != s->scanned.load(std::memory_order_relaxed)) s->scanned.store(*to, std::memory_order_release);
}
// svc_scan for rings that carry runs: the budget is max_slots RECORD SLOTS (a run of k slots counts k) and a run is taken whole or
// left for the next batch (an empty batch takes any run: k <= 16).  Continuation slots are noted as SVC_OP_CONT without reading
// their ready words (the head's release store covers them).  *nslots / *nbytes: record slots / stored bytes taken so far.
template <class H>
static inline void svc_scan_run(H* s, const uint64_t taken, uint64_t* to, uint32_t* nrec, uint32_t* nslots, uint64_t* nbytes,
                                uint32_t* kinds, const uint32_t max_slots) {
    while (*to - taken < SVC_MAX_OPS) {
        const uint32_t slot = (uint32_t)(*to & (SVC_SLOTS - 1u));
        const uint32_t rw = s->ready[slot].load(std::memory_order_acquire);
        if ((rw >> 2) != (uint32_t)(*to / SVC_SLOTS) + 1u) break;
        const uint32_t kd = rw & 3u;
        uint32_t k = 1;
        if (kd == SVC_OP_RECORD) {
            const uint32_t len = __atomic_load_n(&s->lens[slot], __ATOMIC_RELAXED);
            k = svc_run_slots(len);
            if (*nslots + k > max_slots || *to - taken + k > SVC_MAX_OPS) break;
            (*nrec)++; *nslots += k; *nbytes += len;
        }
        for (uint32_t j = 0; j < k; ++j) {
            const uint64_t p = *to + j - taken;
            kinds[p >> 4] |= (j ? (uint32_t)SVC_OP_CONT : kd) << ((p & 15u) * 2u);
        }
        *to += k;
    }
    if (*to != s->scanned.load(std::memory_order_relaxed)) s->scanned.store(*to, std::memory_order_release);
}
