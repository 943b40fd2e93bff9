// agr_svc.cu — the service kernel of the single-request front end (see agr_svc.h for the protocol).
//
// ONE resident CTA of SVC_MAX_OPS threads.  It polls the dispatcher's descriptor ring in pinned host memory, and for every
// batch (<= 512 operations that were in flight at the same time) runs, in this order:
//   records   (proxyToAgentHandler + StoreRequest, server.go:493-541, requests.go:64-117): payloads are pulled out of host
//             memory into shared memory, copied to their slab rows with the record checksum (warp per record), decided one
//             record per thread with the same k1_begin / k1_finish / k1_post_one as the batch kernels;
//   outcomes  (RoundTrip -> StoreResponse / MarkRequestFailed, server.go:583-615, requests.go:120-275): k2_link_one /
//             k2_apply_one of agr_device.cuh behind CTA barriers, and an ordered append to the completed / failed logs
//             (a block scan instead of k2_append's decoupled look-back: the whole batch is in this CTA);
// then writes verdict, Request.ID, row and result code of every operation back to host memory, fences, and flips the
// per-slot done words the callers spin on.  Integer / byte work only; nothing here is on a tensor core.
// Two instantiations: fixed-stride 512 B records (one slot each), and variable-length records (AGR_CFG_VARLEN: a record's run of
// k = ceil(len / 512) slots lands in k consecutive stage slots and goes to the byte slab at the batch's base + the sum of the
// stored lengths before it, as k1_ingest_var would put it).
#include "agr_device.cuh"
#include "agr_svc.h"

// Warp-specialised, two stages deep: four LOADER warps poll the descriptor ring and pull batch k + 1 out of host memory (two
// PCIe round trips) into one shared-memory stage while twelve WORKER warps decide batch k from the other stage, so the kernel's
// cycle is max(poll + pull, decide) instead of their sum.  Named barriers hand a stage over: FULL[s] (loaders arrive, workers
// wait) and FREE[s] (workers arrive, loaders wait).
#define SVC_LOADERS 128u
#define SVC_WORKERS 384u
#define SVC_THREADS (SVC_LOADERS + SVC_WORKERS)
#define SVC_MAX_RECS 128u                                   // records per batch that fit one shared-memory stage
#define SVC_STAGE (SVC_MAX_RECS * 512u + SVC_MAX_OPS * 64u) // 80 KiB
#define SVC_SMEM (2u * SVC_STAGE)                           // 160 KiB
// variable-length records: behind each stage, per record its stored length, its byte offset in the batch and its first stage
// slot, then the batch's record-slot count and the loader warps' partial sums (a maximal 8192 B record is 16 of the 128 slots)
#define SVC_VX_LEN 0u
#define SVC_VX_VOFF (SVC_MAX_RECS * 4u)
#define SVC_VX_FIRST (SVC_MAX_RECS * 8u)
#define SVC_VX_MISC (SVC_MAX_RECS * 10u)
#define SVC_STAGE_VAR (SVC_STAGE + SVC_MAX_RECS * 10u + 32u)   // 81.3 KiB
#define SVC_SMEM_VAR (2u * SVC_STAGE_VAR)                   // 162.6 KiB
#define BAR_FULL0 1
#define BAR_FREE0 3
#define BAR_WORK 5
#define BAR_LOAD 6

__device__ __forceinline__ uint4 ld_sys_v4(const void* p) {                 // host memory, written by CPUs: never cached
    uint4 r;
    asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
    return r;
}
__device__ __forceinline__ uint32_t ld_sys_u32(const volatile uint32_t* p) { return *p; }
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ uint4 lds_v4(const uint8_t* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ void st_res(svc_res* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {   // one 16-byte write
    asm volatile("st.volatile.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// check word of a descriptor (the dispatcher computes the same over the same 62 words, agr_svc_desc_check below)
__host__ __device__ __forceinline__ unsigned long long svc_mix_word(uint32_t w, uint32_t i) {
    return ((unsigned long long)w + 0x9e3779b97f4a7c15ULL * (i + 1u)) * (0xbf58476d1ce4e5b9ULL + 2ULL * i);
}

template <bool VAR>
__global__ void __launch_bounds__(SVC_THREADS, 1)
k_svc(const agr_dev d0, const svc_dev v, const agr_k2_scratch k2, const unsigned long long first_seq) {
    constexpr uint32_t STAGE = VAR ? SVC_STAGE_VAR : SVC_STAGE;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(16) uint32_t s_dw[2][64];           // the accepted descriptors, as words
    __shared__ uint32_t s_go[2], s_nout[2];
    __shared__ uint16_t s_rec_op[2][SVC_MAX_RECS], s_out_op[2][SVC_MAX_OPS];
    __shared__ uint32_t s_wc[12], s_wf[12];
    __shared__ unsigned long long s_logbase[2];
    __shared__ long long s_cyc[2];                           // loader's clock64 accounting: waiting for a batch, pulling payloads
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;

    if (tid < SVC_LOADERS) {
        // ================================================================== LOADERS: poll, map, pull
        unsigned long long last_work = globaltimer_ns(), polls = 0;
        long long c_wait = 0, c_load = 0, c0 = clock64();
        for (unsigned long long seq = first_seq;; ++seq) {
            const uint32_t st = (uint32_t)(seq & 1ULL);
            if (seq >= first_seq + 2ULL) bar_sync(BAR_FREE0 + (int)st, SVC_THREADS);      // the workers are done with batch seq - 2
            uint8_t* s_rec = smem + st * STAGE;
            uint8_t* s_out = s_rec + SVC_MAX_RECS * 512u;
            uint8_t* s_vx = s_rec + SVC_STAGE;                                  // (VAR only)
            uint32_t* vx_len = reinterpret_cast<uint32_t*>(s_vx + SVC_VX_LEN);
            uint32_t* vx_voff = reinterpret_cast<uint32_t*>(s_vx + SVC_VX_VOFF);
            uint16_t* vx_first = reinterpret_cast<uint16_t*>(s_vx + SVC_VX_FIRST);
            uint32_t* vx_misc = reinterpret_cast<uint32_t*>(s_vx + SVC_VX_MISC);   // [0] record slots, [4..7] loader warp sums
            if (warp == 0) {
                const svc_desc* dp = v.desc + (seq % SVC_DESCS);
                uint32_t go = 2u;                                               // 2 = keep polling
                bool stop_seen = false;
                while (go == 2u) {
                    uint4 w = make_uint4(0, 0, 0, 0);
                    uint32_t stop = 0;
                    if (lane < 16u) w = ld_sys_v4(reinterpret_cast<const uint8_t*>(dp) + lane * 16u);
                    else if (lane == 16u) stop = ld_sys_u32(&v.ctl->stop);
                    unsigned long long part = 0;
                    if (lane < 16u) {
                        const uint32_t b = lane * 4u;
                        if (lane != 15u) part = svc_mix_word(w.x, b) ^ svc_mix_word(w.y, b + 1) ^ svc_mix_word(w.z, b + 2) ^ svc_mix_word(w.w, b + 3);
                        else part = svc_mix_word(w.z, b + 2) ^ svc_mix_word(w.w, b + 3);     // lane 15: .x,.y = check, .z,.w = seq
                    }
                    const unsigned long long sum = pack64(__reduce_xor_sync(FULL, (uint32_t)part), __reduce_xor_sync(FULL, (uint32_t)(part >> 32)));
                    const unsigned long long got = pack64(__shfl_sync(FULL, w.z, 15), __shfl_sync(FULL, w.w, 15));
                    const unsigned long long chk = pack64(__shfl_sync(FULL, w.x, 15), __shfl_sync(FULL, w.y, 15));
                    const uint32_t stop_now = __shfl_sync(FULL, stop, 16);
                    polls++;
                    if (got == seq && chk == sum) {
                        if (lane < 16u) { s_dw[st][lane * 4u] = w.x; s_dw[st][lane * 4u + 1] = w.y; s_dw[st][lane * 4u + 2] = w.z; s_dw[st][lane * 4u + 3] = w.w; }
                        go = 1u;
                    } else if (stop_seen) {
                        go = 0u;                                                // stop was set and one more poll found nothing: leave
                    } else if (stop_now) {
                        stop_seen = true;                                       // batches published before the stop must still run
                    } else if (globaltimer_ns() - last_work > v.idle_ns) {
                        go = 3u;                                                // safety: nobody feeds us and nobody stopped us
                    }
                }
                __syncwarp();
                uint32_t nout = 0;
                if (go == 1u) {
                    // op -> (record i | outcome j) maps: thirty-two ops per step, running offsets.  Variable-length records:
                    // s_rec_op maps STAGE SLOTS (record and continuation slots in ring order) to ops, vx_first record -> slot
                    const svc_desc& D = *reinterpret_cast<const svc_desc*>(s_dw[st]);
                    uint32_t br = 0, bo = 0, bs = 0;
                    const uint32_t lt = (1u << lane) - 1u;
                    for (uint32_t base = 0; base < D.count; base += 32u) {
                        const uint32_t op = base + lane;
                        const uint32_t kind = (op < D.count) ? ((D.kinds[op >> 4] >> ((op & 15u) * 2u)) & 3u) : 0u;
                        const uint32_t mr = __ballot_sync(FULL, kind == SVC_OP_RECORD), mo = __ballot_sync(FULL, kind == SVC_OP_OUTCOME);
                        if constexpr (VAR) {
                            const bool in_run = kind == SVC_OP_RECORD || kind == SVC_OP_CONT;
                            const uint32_t ms = __ballot_sync(FULL, in_run), js = bs + __popc(ms & lt);
                            if (in_run) s_rec_op[st][js] = (uint16_t)op;
                            if (kind == SVC_OP_RECORD) vx_first[br + __popc(mr & lt)] = (uint16_t)js;
                            bs += __popc(ms);
                        } else {
                            if (kind == SVC_OP_RECORD) s_rec_op[st][br + __popc(mr & lt)] = (uint16_t)op;
                        }
                        if (kind == SVC_OP_OUTCOME) s_out_op[st][bo + __popc(mo & lt)] = (uint16_t)op;
                        br += __popc(mr); bo += __popc(mo);
                    }
                    nout = bo;
                    if constexpr (VAR) { if (lane == 0) vx_misc[0] = bs; }
                    last_work = globaltimer_ns();
                }
                if (lane == 0) {
                    s_go[st] = go; s_nout[st] = nout;
                    if (go != 1u) v.ctl->heartbeat = polls;
                    const long long c = clock64(); c_wait += c - c0; c0 = c;
                }
            }
            bar_sync(BAR_LOAD, SVC_LOADERS);
            const uint32_t go = s_go[st];
            if (go == 1u) {
                // pull the payloads out of host memory: eight 16-byte loads in flight per thread
                const svc_desc& D = *reinterpret_cast<const svc_desc*>(s_dw[st]);
                const uint32_t rec_chunks = (VAR ? vx_misc[0] : D.n_records) * 32u, total = rec_chunks + s_nout[st] * 4u;
                const unsigned long long from = D.from;
                uint32_t len = 0;                                               // (VAR) record tid's length word: same round trip
                if constexpr (VAR) {
                    if (tid < D.n_records) len = ld_sys_u32(v.lens + ((from + s_rec_op[st][vx_first[tid]]) & (SVC_SLOTS - 1u)));
                }
                for (uint32_t cb = tid; cb < total; cb += SVC_LOADERS * 8u) {
                    uint4 val[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const uint32_t c = cb + (uint32_t)u * SVC_LOADERS;
                        if (c < total) {
                            const bool isrec = c < rec_chunks;
                            const uint32_t item = isrec ? (c >> 5) : ((c - rec_chunks) >> 2), ch = isrec ? (c & 31u) : ((c - rec_chunks) & 3u);
                            const uint32_t op = isrec ? s_rec_op[st][item] : s_out_op[st][item];
                            val[u] = ld_sys_v4(v.payload + (size_t)((from + op) & (SVC_SLOTS - 1u)) * SVC_PAYLOAD + ch * 16u);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const uint32_t c = cb + (uint32_t)u * SVC_LOADERS;
                        if (c < total) {
                            const bool isrec = c < rec_chunks;
                            uint8_t* dst = isrec ? s_rec + (size_t)c * 16u : s_out + (size_t)(c - rec_chunks) * 16u;
                            *reinterpret_cast<uint4*>(dst) = val[u];
                        }
                    }
                }
                if constexpr (VAR) {                                            // byte offsets: exclusive scan of the lengths
                    uint32_t x = len;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(FULL, x, o); if ((int)lane >= o) x += y; }
                    if (lane == 31u) vx_misc[4 + warp] = x;
                    bar_sync(BAR_LOAD, SVC_LOADERS);
                    uint32_t pre = 0;
                    for (uint32_t w = 0; w < warp; ++w) pre += vx_misc[4 + w];
                    if (tid < D.n_records) { vx_len[tid] = len; vx_voff[tid] = pre + x - len; }
                }
                if (tid == 0) { const long long c = clock64(); c_load += c - c0; c0 = c; s_cyc[0] = c_wait; s_cyc[1] = c_load; }
            }
            __threadfence_block();
            bar_arrive(BAR_FULL0 + (int)st, SVC_THREADS);                       // the stage is full (or says "leave")
            if (go != 1u) return;
        }
    }

    // ====================================================================== WORKERS: decide, answer
    const uint32_t wt = tid - SVC_LOADERS, wwarp = wt >> 5;
    long long c_work = 0;
    for (unsigned long long seq = first_seq;; ++seq) {
        const uint32_t st = (uint32_t)(seq & 1ULL);
        bar_sync(BAR_FULL0 + (int)st, SVC_THREADS);
        const uint32_t go = s_go[st];
        if (go != 1u) {
            if (wt == 0) {
                __threadfence_system();
                v.ctl->state = (go == 3u) ? 2u : 0u;
            }
            return;
        }
        const long long cw0 = clock64();
        const uint8_t* s_rec = smem + st * STAGE;
        const uint8_t* s_out = s_rec + SVC_MAX_RECS * 512u;
        const uint32_t* vx_len = reinterpret_cast<const uint32_t*>(s_rec + SVC_STAGE + SVC_VX_LEN);     // (VAR only)
        const uint32_t* vx_voff = reinterpret_cast<const uint32_t*>(s_rec + SVC_STAGE + SVC_VX_VOFF);
        const uint16_t* vx_first = reinterpret_cast<const uint16_t*>(s_rec + SVC_STAGE + SVC_VX_FIRST);
        const svc_desc& D = *reinterpret_cast<const svc_desc*>(s_dw[st]);
        const uint32_t nrec = D.n_records, nout = s_nout[st];
        const unsigned long long from = D.from;
        agr_dev d = d0;                                                          // this batch's view of the live window
        d.tail = D.tail; d.head_l = D.head_l; d.tail_phys = D.tail_phys; d.idx_base = D.idx_base; d.dupfix = v.dupfix;
        const uint32_t lt = (1u << lane) - 1u;

        // ------------------------------------------------------------------ records: slab rows + checksum (warp per record)
        if constexpr (VAR) {
            // lane = 16 B chunk, looping over records longer than 512 B; then the continuation cells' tags, fenced before the
            // head's answer (which goes out after the barrier below): the collector sets SVC_COLLECTED in every cell of the run
            // once it has seen the head's, and a late tag store would take it away again
            for (uint32_t i = wwarp; i < nrec; i += SVC_WORKERS / 32u) {
                const uint32_t rid = D.first_p + i, len = vx_len[i], j0 = vx_first[i];
                const uint8_t* src = s_rec + (size_t)j0 * 512u;
                uint8_t* dst = d.slab + D.vbase + vx_voff[i];
                uint32_t c0 = 0, c1 = 0;
                for (uint32_t c = lane; c < (len >> 4); c += 32u) {
                    const uint4 x = lds_v4(src + (size_t)c * 16u);
                    *reinterpret_cast<uint4*>(dst + (size_t)c * 16u) = x;
                    c0 += x.x + x.y + x.z + x.w;
                    c1 += (4u * c + 1u) * x.x + (4u * c + 2u) * x.y + (4u * c + 3u) * x.z + (4u * c + 4u) * x.w;
                }
                c0 = __reduce_add_sync(FULL, c0); c1 = __reduce_add_sync(FULL, c1);
                if (lane == 0) d.cksum[rid] = agr_cksum_pack(c0, c1);
                const uint32_t k = (len + SVC_PAYLOAD - 1u) / SVC_PAYLOAD;
                if (k > 1u) {                                                    // warp-uniform
                    if (lane >= 1u && lane < k) {
                        const unsigned long long slot_abs = from + s_rec_op[st][j0 + lane];
                        st_res(v.res + (slot_abs & (SVC_SLOTS - 1u)), 0u, 0u, 0u, svc_tag(slot_abs) << 16);
                    }
                    __threadfence_system();
                }
            }
        } else {
            for (uint32_t i = wwarp; i < nrec; i += SVC_WORKERS / 32u) {
                const uint32_t rid = D.first_p + i;
                const uint4 x = lds_v4(s_rec + (size_t)i * 512u + lane * 16u);
                *reinterpret_cast<uint4*>(d.slab + (size_t)rid * AGR_REC + lane * 16u) = x;
                uint32_t c0 = x.x + x.y + x.z + x.w;
                uint32_t c1 = (4u * lane + 1u) * x.x + (4u * lane + 2u) * x.y + (4u * lane + 3u) * x.z + (4u * lane + 4u) * x.w;
                c0 = __reduce_add_sync(FULL, c0); c1 = __reduce_add_sync(FULL, c1);
                if (lane == 0) d.cksum[rid] = agr_cksum_pack(c0, c1);
            }
        }
        // ------------------------------------------------------------------ records: decision chain, one record per thread
        uint32_t lc[K1_NLC + 1];
#pragma unroll
        for (int c = 0; c <= K1_NLC; ++c) lc[c] = 0;
        if (wt < nrec) {
            const uint8_t* hp = s_rec + (size_t)(VAR ? vx_first[wt] : wt) * 512u;
            const uint4 h0 = lds_v4(hp), h1 = lds_v4(hp + 16), h2 = lds_v4(hp + 32), h3 = lds_v4(hp + 48), h4 = lds_v4(hp + 64), h5 = lds_v4(hp + 80);
            const uint32_t rid = D.first_p + wt;
            k1_ctx cx;
            k1_begin(d, k1_agent_issue(d, h2, h3), h0, h1, h2, h3, h4, h5.x, (VAR ? vx_len[wt] : AGR_REC) - AGR_OFF_PAYLOAD, 0ULL, cx);
            const k1_result r = k1_finish(d, rid, h1, h5, cx, lc);
            d.state[rid] = r.state;
            d.route[rid] = r.route;
            if constexpr (VAR) {                                                  // the row words k1_ingest_var leaves (its TTL
                d.voff[rid] = D.vbase + vx_voff[wt];                              // bounds are agr_expire's: k1v_note_time)
                d.vlen[rid] = vx_len[wt];
            } else if ((r.state & ST_STORED) && (d.cfg_flags & AGR_CFG_RING)) {   // TTL bookkeeping (see k1_note_time)
                unsigned long long t = pack64(h4.x, h4.y);
                atomicMin(d.cmin + rid / AGR_CHUNK_ROWS, t ? t : 1ULL);
                d.mtime[rid] = t;
            }
        }
        __threadfence_block();
        bar_sync(BAR_WORK, SVC_WORKERS);
        if (nrec) {
            const uint32_t dupfix = __ldcg(v.dupfix);
            int delta[3] = {0, 0, 0};
            if (wt < nrec) {
                const uint32_t rid = D.first_p + wt;
                const uint32_t r = k1_post_one(d, rid, dupfix, delta);
                const unsigned long long slot_abs = from + s_rec_op[st][VAR ? vx_first[wt] : wt], lrow = D.first_l + wt;
                const uint2 vw = k1_verdict_word(r);
                st_res(v.res + (slot_abs & (SVC_SLOTS - 1u)), vw.x, vw.y, (uint32_t)lrow, (uint32_t)((lrow >> 32) & 0xffffu) | (svc_tag(slot_abs) << 16));
            }
            k1_post_flush(d, delta, (int)lane);
#pragma unroll
            for (int c = 0; c < K1_NLC; ++c) {
                const uint32_t t = __reduce_add_sync(FULL, lc[c]);
                if (lane == 0 && t) atomicAdd(&d.ctr[c], (unsigned long long)t);
            }
            bar_sync(BAR_WORK, SVC_WORKERS);
            if (wt == 0 && dupfix) *v.dupfix = 0u;
        }

        // ------------------------------------------------------------------ outcomes: link, apply, ordered append
        if (nout) {                                                               // nout is uniform over the workers
            if (wt < nout) {
                const uint8_t* o = s_out + (size_t)wt * 64u;
                k2_link_one(d, k2, wt, lds_v4(o), lds_v4(o + 16), lds_v4(o + 32), lds_v4(o + 48));
            }
            __threadfence_block();
            bar_sync(BAR_WORK, SVC_WORKERS);
            uint32_t cnt[3] = {0u, 0u, 0u};
            if (wt < nout) k2_apply_one(d, k2, wt, cnt);
#pragma unroll
            for (int k = 0; k < 3; ++k) cnt[k] = __reduce_add_sync(FULL, cnt[k]);
            if (lane == 0) {
                if (cnt[0]) atomicAdd(&d.ctr[C_COMPLETIONS], (unsigned long long)cnt[0]);
                if (cnt[1]) atomicAdd(&d.ctr[C_FAILURES], (unsigned long long)cnt[1]);
                if (cnt[2]) atomicAdd(&d.ctr[C_DEAD_LETTERED], (unsigned long long)cnt[2]);
            }
            if (wt == 0) { s_logbase[0] = d.log_len[0]; s_logbase[1] = d.log_len[1]; }
            __threadfence_block();
            bar_sync(BAR_WORK, SVC_WORKERS);
            const uint32_t eff = (wt < nout) ? (uint32_t)__ldcg(&k2.eff[wt]) : 0u;
            const uint32_t bc = __ballot_sync(FULL, eff & 1u), bf = __ballot_sync(FULL, eff & 2u);
            if (lane == 0) { s_wc[wwarp] = __popc(bc); s_wf[wwarp] = __popc(bf); }
            bar_sync(BAR_WORK, SVC_WORKERS);
            uint32_t pc = 0, pf = 0, tc = 0, tf = 0;
#pragma unroll
            for (int w = 0; w < (int)(SVC_WORKERS / 32u); ++w) { if ((uint32_t)w < wwarp) { pc += s_wc[w]; pf += s_wf[w]; } tc += s_wc[w]; tf += s_wf[w]; }
            if (eff) {
                const uint32_t rid = k2.ops[wt].rid;
                if (eff & 1u) { const unsigned long long p = s_logbase[0] + pc + __popc(bc & lt); if (p < d.log_cap) d.completed_log[p] = rid; }
                if (eff & 2u) { const unsigned long long p = s_logbase[1] + pf + __popc(bf & lt); if (p < d.log_cap) d.failed_log[p] = rid; }
            }
            if (wt == 0 && (tc | tf)) {
                unsigned long long nc = s_logbase[0] + tc, nf = s_logbase[1] + tf;
                if (nc > d.log_cap || nf > d.log_cap) {
                    atomicAdd(&d.ctr[C_LOG_OVERFLOW], 1ULL);
                    if (nc > d.log_cap) nc = d.log_cap;
                    if (nf > d.log_cap) nf = d.log_cap;
                }
                d.log_len[0] = nc; d.log_len[1] = nf;
            }
            // the outcomes' result codes (the records' verdicts went out as soon as they were final)
            if (wt < nout) {
                const unsigned long long slot_abs = from + s_out_op[st][wt];
                st_res(v.res + (slot_abs & (SVC_SLOTS - 1u)), (uint32_t)k2.results[wt], 0u, 0u, svc_tag(slot_abs) << 16);
            }
        }
        bar_sync(BAR_WORK, SVC_WORKERS);                                         // everything of the stage has been read
        c_work += clock64() - cw0;
        if (wt == 0) {
            v.ctl->done_seq = seq;
            v.ctl->cyc_wait = s_cyc[0]; v.ctl->cyc_load = s_cyc[1]; v.ctl->cyc_work = c_work; v.ctl->cyc_publish = 0;
        }
        bar_arrive(BAR_FREE0 + (int)st, SVC_THREADS);                            // the loaders may refill it
    }
}

cudaError_t agr_launch_svc(const agr_dev& d, const svc_dev& v, const agr_k2_scratch& k2, unsigned long long next_seq, bool var, cudaStream_t st) {
    static bool attr_done[2] = {false, false};
    const uint32_t smem = var ? SVC_SMEM_VAR : SVC_SMEM;
    if (!attr_done[var]) {
        cudaError_t e = cudaFuncSetAttribute(var ? k_svc<true> : k_svc<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        attr_done[var] = true;
    }
    if (var) k_svc<true><<<1, SVC_THREADS, smem, st>>>(d, v, k2, next_seq);
    else k_svc<false><<<1, SVC_THREADS, smem, st>>>(d, v, k2, next_seq);
    return cudaGetLastError();
}

// host side of the descriptor check (same words, same mix)
unsigned long long agr_svc_desc_check(const svc_desc* dsc) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(dsc);
    unsigned long long s = 0;
    for (uint32_t i = 0; i < 64u; ++i) if (i != 60u && i != 61u) s ^= svc_mix_word(w[i], i);
    return s;
}
