// ring_sim_var.cpp — the run-aware callers' side of the single-request ring (csrc/agr_ring.hpp: svc_submit_run, svc_release_run,
// svc_scan_run) against a stand-in for the dispatcher and the service kernel, on the CPU.  Variable-length records take runs of
// 1 .. 16 slots (96 .. 8192 B), mixed with one-slot operations (svc_submit_one).  Checks:
//   * every operation handed over is answered exactly once, with an answer computed from ALL the slots of its run (a continuation
//     slot overwritten before the run was consumed shows up as a wrong answer);
//   * the stand-in consumes runs whole (a batch never ends inside a run) and answers every cell of a run, continuation cells first;
//   * ticket holders that together hold more tickets than the ring has slots finish; blocking callers and ticket callers share one
//     ring; runs cross the ring's end.
// usage: ring_sim_var <blocking threads> <ticket threads> <tickets in flight per ticket thread> <operations per thread> [service delay us]
// prints one JSON line; exit code 0 = every check passed.  Test infrastructure (tests/test_ring_sim_var.py), no CUDA.
#include <stdio.h>
#include <stdlib.h>
#include <chrono>
#include <thread>
#include <vector>
#include "../agentainer-lab_b200/csrc/agr_ring.hpp"

struct sim_host {
    svc_res* res = nullptr; uint8_t* payload = nullptr; uint32_t* lens = nullptr;
    std::atomic<uint32_t>* ready = nullptr;
    uint32_t spin_cpus = 2;
    std::atomic<bool> sleeping{false};
    alignas(64) std::atomic<uint64_t> head{0};
    alignas(64) std::atomic<uint32_t> waiters{0};
    alignas(64) std::atomic<uint64_t> scanned{0};
    std::mutex smu; std::condition_variable scv;
};

static inline uint64_t mix(uint64_t x) { x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; return x ^ (x >> 33); }
static uint64_t digest(const uint8_t* p, uint32_t len) {          // over every 8-byte word of the record
    uint64_t h = len;
    for (uint32_t o = 0; o < len; o += 8) { uint64_t w; memcpy(&w, p + o, 8); h = mix(h ^ w) + o; }
    return h;
}
// a record of len bytes whose every 16-byte chunk depends on the token
static void fill(uint8_t* p, uint32_t len, uint64_t token) {
    for (uint32_t c = 0; c < len / 16u; ++c) { const uint64_t a = mix(token + c), b = mix(a); memcpy(p + 16 * c, &a, 8); memcpy(p + 16 * c + 8, &b, 8); }
}

int main(int argc, char** argv) {
    const int nb = argc > 1 ? atoi(argv[1]) : 4, nt = argc > 2 ? atoi(argv[2]) : 4;
    const uint32_t inflight = argc > 3 ? (uint32_t)atoi(argv[3]) : 512u;
    const uint64_t per_thread = argc > 4 ? strtoull(argv[4], nullptr, 10) : 100000ULL;
    const int delay_us = argc > 5 ? atoi(argv[5]) : 0;
    sim_host S;
    S.res = (svc_res*)aligned_alloc(64, sizeof(svc_res) * SVC_SLOTS); memset((void*)S.res, 0, sizeof(svc_res) * SVC_SLOTS);
    S.payload = (uint8_t*)aligned_alloc(64, (size_t)SVC_SLOTS * SVC_PAYLOAD); memset(S.payload, 0, (size_t)SVC_SLOTS * SVC_PAYLOAD);
    S.lens = (uint32_t*)aligned_alloc(64, sizeof(uint32_t) * SVC_SLOTS); memset(S.lens, 0, sizeof(uint32_t) * SVC_SLOTS);
    S.ready = new std::atomic<uint32_t>[SVC_SLOTS];
    for (uint32_t i = 0; i < SVC_SLOTS; ++i) S.ready[i].store(0);
    std::atomic<bool> quit{false};
    std::atomic<uint64_t> served{0}, skipped{0}, bad{0}, eagain{0}, done_ops{0}, crossed{0}, torn{0}, maxrun{0};

    // dispatcher + service kernel in one thread: the dispatcher's own run-aware scan (128 record slots per batch, like
    // svc_dispatcher on a variable-length engine), then every real operation answered like k_svc does
    std::thread service([&] {
        uint64_t to = 0;
        std::vector<uint8_t> rec(8192);
        while (!quit.load(std::memory_order_acquire)) {
            const uint64_t from = to;
            uint32_t nrec = 0, nslots = 0, kinds[SVC_MAX_OPS / 16] = {0};
            uint64_t nbytes = 0;
            svc_scan_run(&S, from, &to, &nrec, &nslots, &nbytes, kinds, 128u);
            if (to == from) { std::this_thread::yield(); continue; }
            if (nslots > 128u) torn++;
            if (delay_us) std::this_thread::sleep_for(std::chrono::microseconds(delay_us));     // the batch is "on the GPU"
            auto kind_at = [&](uint64_t a) { return (kinds[(a - from) >> 4] >> (((a - from) & 15u) * 2u)) & 3u; };
            uint64_t got_bytes = 0;
            for (uint64_t a = from; a < to; ++a) {
                const uint32_t slot = (uint32_t)(a & (SVC_SLOTS - 1u));
                const uint32_t kind = kind_at(a);
                if (kind == SVC_OP_SKIP) { skipped++; continue; }
                if (kind == SVC_OP_CONT) continue;                                       // answered with its head
                uint64_t ans;
                if (kind == SVC_OP_RECORD) {
                    const uint32_t len = __atomic_load_n(&S.lens[slot], __ATOMIC_RELAXED), k = svc_run_slots(len);
                    got_bytes += len;
                    if (a + k > to) { torn++; continue; }                                // a batch ended inside a run
                    for (uint32_t j = 1; j < k; ++j) if (kind_at(a + j) != SVC_OP_CONT) torn++;
                    for (uint32_t j = 0; j < k; ++j) {                                   // the loaders: slot by slot
                        const uint32_t n = j + 1u == k ? len - j * SVC_PAYLOAD : SVC_PAYLOAD;
                        memcpy(rec.data() + (size_t)j * SVC_PAYLOAD, S.payload + (size_t)((a + j) & (SVC_SLOTS - 1u)) * SVC_PAYLOAD, n);
                    }
                    if (slot + k > SVC_SLOTS) crossed++;
                    if (k > maxrun.load(std::memory_order_relaxed)) maxrun.store(k, std::memory_order_relaxed);
                    ans = mix(digest(rec.data(), len) ^ a);
                    for (uint32_t j = 1; j < k; ++j)                                     // continuation cells: tag only, first
                        __atomic_store_n(&S.res[(a + j) & (SVC_SLOTS - 1u)].w[3], svc_tag(a + j) << 16, __ATOMIC_RELEASE);
                } else {
                    uint64_t token; memcpy(&token, S.payload + (size_t)slot * SVC_PAYLOAD, 8);
                    ans = mix(token ^ a);
                }
                svc_res* r = S.res + slot;
                __atomic_store_n(&r->w[0], (uint32_t)ans | 1u, __ATOMIC_RELAXED); __atomic_store_n(&r->w[1], (uint32_t)(ans >> 32), __ATOMIC_RELAXED);
                __atomic_store_n(&r->w[2], (uint32_t)kind, __ATOMIC_RELAXED);
                __atomic_store_n(&r->w[3], svc_tag(a) << 16, __ATOMIC_RELEASE);
                served++;
            }
            if (got_bytes != nbytes) torn++;
        }
    });

    auto check = [&](uint64_t a, uint64_t want, const svc_answer& r) {
        const uint64_t ans = mix(want ^ a);
        if (r.w0 != ((uint32_t)ans | 1u) || r.w1 != (uint32_t)(ans >> 32)) bad++;
    };
    // record lengths: every run length 1 .. 16 occurs (96 B .. 8192 B, multiples of 16)
    auto length_of = [](uint64_t token) { return (uint32_t)(96u + 16u * (uint32_t)(token % ((8192u - 96u) / 16u + 1u))); };
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<std::thread> ths;
    for (int t = 0; t < nb; ++t) ths.emplace_back([&, t] {                              // blocking callers: a record, then an outcome
        std::vector<uint8_t> rec(8192);
        alignas(16) uint8_t item[64];
        for (uint64_t i = 0; i < per_thread; ++i) {
            const uint64_t token = mix(((uint64_t)t << 40) | i);
            uint64_t a;
            if (i & 1) {
                memset(item, 0, sizeof item); memcpy(item, &token, 8);
                while (!svc_submit_one(&S, SVC_OP_OUTCOME, item, sizeof item, &a)) {}
                svc_answer r; svc_wait(&S, a, &r);
                check(a, token, r);
                svc_release(&S, a);
            } else {
                const uint32_t len = length_of(token);
                fill(rec.data(), len, token);
                while (!svc_submit_run(&S, rec.data(), len, &a)) {}                      // the blocking call draws again
                svc_answer r; svc_wait(&S, a, &r);
                check(a, digest(rec.data(), len), r);
                svc_release_run(&S, a, svc_run_slots(len));
            }
            done_ops++;
        }
    });
    for (int t = 0; t < nt; ++t) ths.emplace_back([&, t] {                              // ticket callers: a FIFO of parked operations
        struct fl { uint64_t a, want; uint32_t k; };
        std::vector<fl> q(inflight);
        size_t head = 0, count = 0;
        std::vector<uint8_t> rec(8192);
        alignas(16) uint8_t item[64];
        uint64_t issued = 0;
        while (issued < per_thread || count) {
            while (issued < per_thread && count < q.size()) {
                const uint64_t token = mix(((uint64_t)(t + 1000) << 40) | issued);
                uint64_t a, want;
                uint32_t k = 1;
                bool ok;
                if (token % 4 == 0) {                                                    // one-slot operations among the runs
                    memset(item, 0, sizeof item); memcpy(item, &token, 8);
                    ok = svc_submit_one(&S, SVC_OP_OUTCOME, item, sizeof item, &a);
                    want = token;
                } else {
                    const uint32_t len = length_of(token >> 2);
                    fill(rec.data(), len, token);
                    ok = svc_submit_run(&S, rec.data(), len, &a);
                    want = digest(rec.data(), len); k = svc_run_slots(len);
                }
                if (!ok) { eagain++; break; }                                            // AGR_EAGAIN: collect, come again
                q[(head + count) % q.size()] = fl{a, want, k}; count++; issued++;
            }
            uint32_t reaped = 0;
            while (count && reaped < 64) {
                svc_answer r;
                if (!svc_try(&S, q[head].a, &r)) break;
                check(q[head].a, q[head].want, r);
                svc_release_run(&S, q[head].a, q[head].k);
                head = (head + 1) % q.size(); count--; reaped++; done_ops++;
            }
            if (!reaped) _mm_pause();
        }
    });
    for (auto& th : ths) th.join();
    const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    quit.store(true, std::memory_order_release);
    service.join();
    const uint64_t want = (uint64_t)(nb + nt) * per_thread;
    const bool ok = bad.load() == 0 && torn.load() == 0 && done_ops.load() == want && served.load() == want;
    printf("{\"blocking_threads\": %d, \"ticket_threads\": %d, \"inflight\": %u, \"operations\": %llu, \"served\": %llu, \"skipped_slots\": %llu, "
           "\"eagain\": %llu, \"wrong_answers\": %llu, \"torn_runs\": %llu, \"runs_across_ring_end\": %llu, \"longest_run\": %llu, "
           "\"ring_laps\": %.1f, \"seconds\": %.3f, \"ok\": %s}\n",
           nb, nt, inflight, (unsigned long long)done_ops.load(), (unsigned long long)served.load(), (unsigned long long)skipped.load(),
           (unsigned long long)eagain.load(), (unsigned long long)bad.load(), (unsigned long long)torn.load(), (unsigned long long)crossed.load(),
           (unsigned long long)maxrun.load(), (double)S.head.load() / SVC_SLOTS, secs, ok ? "true" : "false");
    return ok ? 0 : 1;
}
