// bench_callers.cpp — the reference's real call pattern at the C-ABI: one OS thread per in-flight HTTP request
// (net/http's goroutine per connection -> proxyToAgentHandler, internal/api/server.go:493-573), every thread doing
//     agr_ingest_ex(n = 1)  ->  [forward]  ->  agr_complete(n = 1)
// i.e. StoreRequest + the routing decision, then StoreResponse (server.go:508-518, 588-594), through the single-request
// front end (AGR_CFG_COMBINE).  Prints ONE JSON object: round trips per second, p50 / p99 latency of a round trip.
// With <inflight> > 0 every thread keeps that many requests in flight through the ticket calls (agr_submit_ingest ->
// agr_poll -> agr_submit_complete -> agr_poll): the goroutine-per-request pattern of a Go host, where a request parks instead
// of pinning an OS thread (INTEGRATION.md).  Every request is still handed over one at a time.
// With a 7th argument the records are VARIABLE-LENGTH (AGR_CFG_VARLEN, BASELINE config 5: bodies log-uniform in [128 B, 4 KB]),
// handed over with agr_ingest_var(n = 1) / agr_submit_ingest_var: "var" through the single-request front end, "var_launch" with
// AGR_CFG_COMBINE off (every call is a launch + a stream sync: what the front end is measured against; blocking calls only).
//   bench_callers <threads> <seconds> [device] [mint|hash] [agents] [inflight per thread, 0 = blocking calls] [var|var_launch]
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <cmath>
#include <string>
#include <thread>
#include <vector>

#include "../../include/agentainer_gpu.h"

static uint64_t splitmix(uint64_t& x) {
    uint64_t z = (x += 0x9e3779b97f4a7c15ULL);
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL; z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
    return z ^ (z >> 31);
}

int main(int argc, char** argv) {
    const int threads = argc > 1 ? atoi(argv[1]) : 64;
    const double seconds = argc > 2 ? atof(argv[2]) : 2.0;
    const int device = argc > 3 ? atoi(argv[3]) : 0;
    const bool mint = !(argc > 4 && strcmp(argv[4], "hash") == 0);
    const int n_agents = argc > 5 ? atoi(argv[5]) : 256;
    const int inflight = argc > 6 ? atoi(argv[6]) : 0;
    const bool var = argc > 7, combine = !(var && strcmp(argv[7], "var_launch") == 0);
    if (var && strcmp(argv[7], "var") != 0 && combine) { fprintf(stderr, "7th argument: var | var_launch\n"); return 2; }
    if (!combine && inflight > 0) { fprintf(stderr, "tickets need the single-request front end (var, not var_launch)\n"); return 2; }
    agr_config cfg; memset(&cfg, 0, sizeof cfg);
    cfg.device = device;
    cfg.slab_rows = 1ull << 26;                         // 64 Mi rows = 32 GiB of slab: ~10 s at 6 M round trips/s
    cfg.max_agents = 1024; cfg.max_batch = 1u << 16; cfg.log_entries = cfg.slab_rows; cfg.resp_bytes = 1 << 20;
    cfg.flags = AGR_CFG_PERSISTENCE | (combine ? AGR_CFG_COMBINE : 0u) | (mint ? AGR_CFG_MINT_IDS : 0u);
    if (var) {
        cfg.slab_rows = 1ull << 25;                     // 32 Mi rows, 48 GiB of byte slab (~1.3 KB a record)
        cfg.log_entries = cfg.slab_rows; cfg.vslab_bytes = 48ull << 30;
        cfg.flags |= AGR_CFG_VARLEN;
    }
    agr_handle* h = nullptr;
    if (agr_create(&cfg, &h) < 0) { fprintf(stderr, "agr_create: %s\n", agr_last_error()); return 2; }
    agr_synth sy; memset(&sy, 0, sizeof sy); sy.seed = 7; sy.n_agents = (uint32_t)n_agents;
    std::vector<std::string> names;
    for (int k = 0; k < n_agents; ++k) {
        char id[AGR_AGENT_ID_BYTES]; agr_synth_agent_id(&sy, (uint32_t)k, id);
        names.emplace_back(id);
        if (agr_set_agent_state(h, id, AGR_AGENT_RUNNING) < 0) { fprintf(stderr, "set_agent_state: %s\n", agr_last_error()); return 2; }
    }
    std::atomic<bool> go{false}, stop{false};
    std::atomic<uint64_t> total{0}, bad{0};
    std::vector<std::vector<uint32_t>> lat(threads);
    std::vector<std::thread> ths;
    for (int t = 0; t < threads; ++t) ths.emplace_back([&, t] {
        // every thread sends the synthetic stream's records (BASELINE's 512 B POST /agent/<id>/chat shape), one per call
        std::vector<agr_record> recs(64);
        agr_synth s2 = sy; s2.seed = 1000 + t;
        agr_synth_fill_host(&s2, 0, 64, recs.data());
        // variable-length form of the same records: header, path | headers, then a body of log-uniform size in [128 B, 4 KB]
        std::vector<std::vector<uint8_t>> vrec(var ? 64 : 0);
        uint64_t xb = 0x9999 + t;
        for (size_t k = 0; k < vrec.size(); ++k) {
            agr_record& r = recs[k];
            const uint32_t body = (uint32_t)std::exp(std::log(128.0) + (double)(splitmix(xb) >> 11) * 0x1.0p-53 * (std::log(4096.0) - std::log(128.0)));
            const uint32_t ph = r.path_len + r.hdr_len, len = 96u + ((ph + body + 15u) & ~15u);
            vrec[k].assign(len, 0);
            r.body_len = body;
            memcpy(vrec[k].data(), &r, 96); memcpy(vrec[k].data() + 96, r.payload, ph);
            for (uint32_t b = 0; b < body; ++b) vrec[k][96 + ph + b] = (uint8_t)(32 + (splitmix(xb) % 95));
        }
        auto set_head = [&](uint32_t k) {                  // request id / seq of recs[k] into its variable-length form
            if (var) memcpy(vrec[k].data(), &recs[k], 96);
        };
        uint64_t x = 0x1234 + t, n = 0;
        auto& my = lat[t]; my.reserve(1 << 20);
        while (!go.load(std::memory_order_acquire)) std::this_thread::yield();
        if (inflight > 0) {
            // Tickets are answered in hand-over order (batch by batch), so the thread keeps its requests in a FIFO and polls only
            // the OLDEST one: a poll that says "not yet" means nothing younger is ready either.
            struct flight { int stage; agr_ticket t; std::chrono::steady_clock::time_point t0; uint32_t rec; };
            std::vector<flight> q((size_t)inflight);
            size_t head = 0, count = 0;                                   // FIFO over q: [head, head + count)
            auto push = [&](const flight& f) { q[(head + count) % q.size()] = f; count++; };
            while (!stop.load(std::memory_order_relaxed)) {
                while (count < q.size()) {                                 // start requests: StoreRequest + routing decision
                    flight f; f.rec = (uint32_t)(n & 63); agr_record& r = recs[f.rec];
                    if (!mint) { uint64_t a = splitmix(x), b = splitmix(x) | 1; memcpy(r.request_id, &a, 8); memcpy(r.request_id + 8, &b, 8); }
                    r.seq = n;
                    set_head(f.rec);
                    f.t0 = std::chrono::steady_clock::now();
                    const int rc = var ? agr_submit_ingest_var(h, vrec[f.rec].data(), (uint32_t)vrec[f.rec].size(), &f.t) : agr_submit_ingest(h, &r, &f.t);
                    if (rc == AGR_EAGAIN) break;
                    if (rc < 0) { bad++; stop.store(true); break; }
                    f.stage = 0; n++;
                    push(f);
                }
                uint32_t reaped = 0;
                while (count && reaped < 64) {
                    flight f = q[head];
                    agr_result res;
                    const int rc = agr_poll(h, f.t, &res);
                    if (rc == AGR_EAGAIN) break;
                    head = (head + 1) % q.size(); count--; reaped++;
                    if (rc < 0 || res.result != 0) { bad++; stop.store(true); break; }
                    if (f.stage == 0) {                                    // forwarded: the agent answered, StoreResponse
                        if (res.verdict.code != AGR_V_FORWARD) { bad++; stop.store(true); break; }
                        agr_outcome o; memset(&o, 0, sizeof o);
                        memcpy(o.request_id, res.request_id, 16); memcpy(o.agent_id, recs[f.rec].agent_id, AGR_AGENT_ID_BYTES);
                        o.kind = AGR_OUT_RESPONSE; o.http_status = 200; o.seq = n;
                        int rc2;
                        // AGR_EAGAIN: the slot drawn still holds somebody's uncollected answer; the next draw is another slot
                        while ((rc2 = agr_submit_complete(h, &o, &f.t)) == AGR_EAGAIN && !stop.load(std::memory_order_relaxed)) {}
                        if (rc2 == AGR_EAGAIN) break;                      // the run is over: this request stays forwarded-but-uncompleted
                        if (rc2 < 0) { bad++; stop.store(true); break; }
                        f.stage = 1;
                        push(f);
                    } else {
                        const auto t1 = std::chrono::steady_clock::now();
                        if (my.size() < my.capacity()) my.push_back((uint32_t)std::chrono::duration_cast<std::chrono::nanoseconds>(t1 - f.t0).count());
                    }
                }
            }
            while (count) { agr_result res; agr_wait(h, q[head].t, &res); head = (head + 1) % q.size(); count--; }   // drain
            total += n;
            return;
        }
        while (!stop.load(std::memory_order_relaxed)) {
            agr_record& r = recs[n & 63];
            if (!mint) { uint64_t a = splitmix(x), b = splitmix(x) | 1; memcpy(r.request_id, &a, 8); memcpy(r.request_id + 8, &b, 8); }
            r.seq = n;
            set_head((uint32_t)(n & 63));
            agr_verdict v; uint8_t id[1][16]; uint64_t first;
            const auto t0 = std::chrono::steady_clock::now();
            int rc;
            if (var) {
                const uint32_t off[2] = {0u, (uint32_t)vrec[n & 63].size()};
                rc = agr_ingest_var(h, vrec[n & 63].data(), off, 1, &v, id, &first);
            } else rc = agr_ingest_ex(h, &r, 1, &v, id, &first);
            if (rc < 0 || v.code != AGR_V_FORWARD) { bad++; break; }
            agr_outcome o; memset(&o, 0, sizeof o);
            memcpy(o.request_id, id[0], 16); memcpy(o.agent_id, r.agent_id, AGR_AGENT_ID_BYTES);
            o.kind = AGR_OUT_RESPONSE; o.http_status = 200; o.seq = n + 1;
            int32_t res = -1;
            if (agr_complete(h, &o, 1, &res) < 0 || res != 0) { bad++; break; }
            const auto t1 = std::chrono::steady_clock::now();
            if (my.size() < my.capacity()) my.push_back((uint32_t)std::chrono::duration_cast<std::chrono::nanoseconds>(t1 - t0).count());
            n++;
        }
        total += n;
    });
    // warm-up: let the dispatcher and the resident kernel come up, then measure
    go.store(true, std::memory_order_release);
    std::this_thread::sleep_for(std::chrono::milliseconds(300));
    for (auto& v : lat) v.clear();                      // (racy by design: warm-up samples may survive; they are few)
    agr_stats s0; agr_stats_get(h, &s0);
    const auto t0 = std::chrono::steady_clock::now();
    std::this_thread::sleep_for(std::chrono::duration<double>(seconds));
    agr_stats s1; agr_stats_get(h, &s1);
    const auto t1 = std::chrono::steady_clock::now();
    stop.store(true);
    for (auto& th : ths) th.join();
    const double secs = std::chrono::duration<double>(t1 - t0).count();
    // every round trip is one stored request + one completion: count them on the ENGINE's side of the boundary
    const double rt = (double)(s1.completions - s0.completions);
    std::vector<uint32_t> all;
    for (auto& v : lat) all.insert(all.end(), v.begin(), v.end());
    std::sort(all.begin(), all.end());
    auto pct = [&](double p) { return all.empty() ? 0.0 : all[(size_t)std::min<double>(all.size() - 1, p * all.size())] / 1000.0; };
    agr_stats s2; agr_stats_get(h, &s2);
    printf("{\"threads\": %d, \"seconds\": %.3f, \"round_trips\": %.0f, \"round_trips_per_s\": %.1f, \"ops_per_s\": %.1f, "
           "\"p50_us\": %.2f, \"p99_us\": %.2f, \"latency_samples\": %zu, \"svc_batches\": %llu, \"ops_per_batch\": %.1f, "
           "\"id_mode\": \"%s\", \"agents\": %d, \"inflight_per_thread\": %d, \"errors\": %llu, \"stored\": %llu, \"completions\": %llu, \"host_cpus\": %u%s}\n",
           threads, secs, rt, rt / secs, 2.0 * rt / secs, pct(0.50), pct(0.99), all.size(),
           (unsigned long long)(s1.svc_batches - s0.svc_batches), (double)(s1.svc_ops - s0.svc_ops) / std::max<double>(1.0, (double)(s1.svc_batches - s0.svc_batches)),
           mint ? "mint" : "hash", n_agents, inflight, (unsigned long long)bad.load(), (unsigned long long)s2.stored, (unsigned long long)s2.completions,
           std::thread::hardware_concurrency(), var ? (combine ? ", \"records\": \"var\"" : ", \"records\": \"var_launch\"") : "");
    agr_destroy(h);
    return bad.load() ? 1 : 0;
}
