// shard.cu -- the prefix/suffix table sharded by key hash over the GPUs of one box (SURVEY.md 8(e), north_star):
// shard g (table.cu, stage_build_table(rank, world)) indexes the keys with key_owner(hash) == g; the reads stay
// replicated.  A window probe of HashTable::hashTableSearch (hashTable.cpp:193-231) becomes a routed query:
//
//   source  route_begin   the window keys of a batch of reads (a slice of phase A, the redo list, or the reads left
//                         for phase C) are derived (utils.cpp:171-207) and bucketed by owner: one contiguous
//                         stream of queries per owner + the map send position -> (read of the batch, window).
//                         A query is the 64-bit key hash (tag probes) or the 128-bit key (verified probes).
//           [all-to-all of the query streams: NCCL over NVLink, sage2_b200/multi.py]
//   owner   shard_answer  one thread per received query probes the shard's sector index and answers with a slot
//                         word without its tag (count | inline entry / run offset); the entry runs of the
//                         2..99-entry buckets are copied into one stream per source, in query order.
//           [all-to-all of the answer words and of the entry streams]
//   source  route_finish  answers are scattered to wslot[read of the batch][window] (run offsets rebased into the
//                         concatenated entry streams): a direct-indexed table of exactly the probes the batch needs.
//
// The search kernels then run unchanged except for stage 1 (search.cu, ROUTED): a coalesced load of wslot instead
// of a random sector probe.  Tag probes are proven by the search kernel itself (first entry of every bucket /
// representative of a masked key); a 24-bit tag collision flags the read, and the flagged reads are routed again
// with verified probes (the owner confirms the key from its copy of the reads, hashTable.cpp:203-220).
#include <stdlib.h>
#include <string.h>
#include "context.h"

namespace sg {

constexpr int RT_WARPS = 8;

__device__ __forceinline__ void ldg256s(const u64 *p, u64 (&v)[4])
{
    asm volatile("ld.global.nc.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v[0]), "=l"(v[1]), "=l"(v[2]), "=l"(v[3]) : "l"(p));
}

// ---- source: keys of a batch, bucketed by owner ------------------------------------------------------------
// Where the stream of every owner goes: dst[g] = first query word of owner g's stream -- local memory (NCCL
// exchange) or the owner's mailbox in PEER memory (the stores then travel over NVLink while the kernel runs);
// qoff[g] = position of the stream in the local send-order map qmap.
struct RouteDst {
    u64 *dst[kMaxWorld];
    u64 qoff[kMaxWorld];
};

// WRITE = false: g_count[g] += queries for owner g.  WRITE = true: g_count[g] is the cursor of owner g's stream
// (starts at 0); a tile of RT_WARPS reads reserves its share with one atomic per owner.
template <bool WRITE>
__global__ void __launch_bounds__(RT_WARPS * 32) route_kernel(const u64 *__restrict__ F, int SW, int SWS, int h, const u32 *__restrict__ ids, u64 first,
                                                              u64 n, u32 wstride, int world, int exact, unsigned long long *__restrict__ g_count,
                                                              const __grid_constant__ RouteDst D, u32 *__restrict__ qmap)
{
    __shared__ u64 sX[RT_WARPS][kMaxWords];
    __shared__ unsigned int tcount[kMaxWorld];
    __shared__ unsigned long long tbase[kMaxWorld];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    u64 *X = sX[warp];
    if (threadIdx.x < kMaxWorld) tcount[threadIdx.x] = 0;
    __syncthreads();
    const u64 ntiles = (n + RT_WARPS - 1) / RT_WARPS;
    for (u64 tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const u64 s = tile * RT_WARPS + warp;
        const bool active = s < n;
        int W = 0;
        if (active) {
            const u64 i = ids ? (u64)ids[s] : first + s;
            for (int w = lane; w < SW; w += 32) X[w] = F[i * SWS + w];
            __syncwarp();
            W = rec_len(X, SW) - h + 1;
        }
        u64 hc0 = 0, hc1 = 0, hc2 = 0, hc3 = 0;        // key hashes of the first four chunks, computed once for both passes
#pragma unroll 1
        for (int pass = 0; pass < (WRITE ? 2 : 1); ++pass) {
            for (int base = 0; base < W; base += 32) {
                const int j = base + lane;
                int g = -1;
                u64 v0 = 0, v1 = 0, hsh = 0;
                if (j < W) {
                    const int ch = base >> 5;
                    const bool cached = WRITE && !exact && pass == 1 && ch < 4;
                    if (cached) hsh = ch == 0 ? hc0 : ch == 1 ? hc1 : ch == 2 ? hc2 : hc3;
                    else {
                        extract_key(X, SW, j, h, v0, v1);
                        hsh = hash_key(v0, v1);
                        if (WRITE && pass == 0) { if (ch == 0) hc0 = hsh; else if (ch == 1) hc1 = hsh; else if (ch == 2) hc2 = hsh; else if (ch == 3) hc3 = hsh; }
                    }
                    g = key_owner(hsh, world);
                }
                const unsigned same = __match_any_sync(0xffffffffu, g);
                const int leader = __ffs(same) - 1;
                unsigned off = 0;
                if (g >= 0 && lane == leader) off = atomicAdd(&tcount[g], (unsigned)__popc(same));
                if (WRITE && pass == 1) {
                    off = __shfl_sync(0xffffffffu, off, leader);
                    if (g >= 0) {
                        const u64 pos = tbase[g] + off + (unsigned)__popc(same & lt_mask);
                        u64 *q = D.dst[g];
                        if (exact) { q[2 * pos] = v0; q[2 * pos + 1] = v1; }
                        else q[pos] = hsh;
                        qmap[D.qoff[g] + pos] = (u32)(s * wstride + (u64)j);
                    }
                }
            }
            if (WRITE && pass == 0) {
                __syncthreads();
                if (threadIdx.x < world) {
                    tbase[threadIdx.x] = atomicAdd(&g_count[threadIdx.x], (unsigned long long)tcount[threadIdx.x]);
                    tcount[threadIdx.x] = 0;
                }
                __syncthreads();
            }
        }
        if (WRITE) {
            __syncthreads();
            if (threadIdx.x < world) tcount[threadIdx.x] = 0;
            __syncthreads();
        }
    }
    if (!WRITE) {
        __syncthreads();
        if (threadIdx.x < world && tcount[threadIdx.x]) atomicAdd(&g_count[threadIdx.x], (unsigned long long)tcount[threadIdx.x]);
    }
}

// ---- owner: answers -------------------------------------------------------------------------------------------
// hashTableSearch on this shard's sector index.  Tag probes take the first slot whose 24-bit tag matches (proven by
// the source's search kernel); verified probes confirm the key from the bucket's first read and skip masked keys.
constexpr u32 kEntryChunk = 1024;     // entries a warp of answer_fused_kernel reserves at a time (one atomic per ~1000 entries)

struct ShardView {
    const u64 *slots;
    u64 nsec;
    const u32 *entries;
    const u64 *F, *RC;
    const uint16_t *len;
    int SW, SWS, h;
};

// answer word of query p (payload = OWNER-side offset for a 2..99-entry bucket, whose length comes back in `run`)
__device__ __forceinline__ u64 answer_one(const ShardView &T, const u64 *__restrict__ queries, u64 p, int exact, u32 &run)
{
    const u64 *slots = T.slots, *F = T.F, *RC = T.RC;
    const u32 *entries = T.entries;
    const uint16_t *len = T.len;
    const u64 nsec = T.nsec;
    const int SW = T.SW, SWS = T.SWS, h = T.h;
    {
        u64 v0 = 0, v1 = 0, hsh;
        if (exact) { v0 = queries[2 * p]; v1 = queries[2 * p + 1]; hsh = hash_key(v0, v1); }
        else hsh = queries[p];
        const u64 tag = slot_tag(hsh);
        u64 answer = 0;
        run = 0;
        bool done = nsec == 0;
        u64 sec = done ? 0 : home_sector(hsh, nsec);
        while (!done) {
            u64 s[4];
            ldg256s(slots + kSlotsPerSector * sec, s);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                if (done) continue;
                const u64 slot = s[t];
                if (slot == 0) { done = true; continue; }
                if (slot_get_tag(slot) != tag) continue;
                const u32 c = slot_get_count(slot);
                const u64 pay = slot_get_payload(slot);
                if (exact) {
                    const u32 ent = (c == 1 || c >= (u32)kHashThreshold) ? (u32)pay : __ldg(&entries[pay]);
                    const u64 rid = ent >> 2;
                    u64 w0, w1;
                    entry_key(F + rid * SWS, RC + rid * SWS, SW, len[rid], h, (int)(ent & 3), w0, w1);
                    if (w0 != v0 || w1 != v1) continue;                     // tag collision: keep probing
                    if (c >= (u32)kHashThreshold) { done = true; continue; }   // masked key reads as absent (hashTable.cpp:203)
                }
                answer = answer_encode(c, pay);
                if (c >= 2 && c < (u32)kHashThreshold) run = c;
                done = true;
            }
            sec = (sec + 1 == nsec) ? 0 : sec + 1;
        }
        return answer;
    }
}

__global__ void __launch_bounds__(256) answer_kernel(const u64 *__restrict__ queries, u64 nq, int exact, const __grid_constant__ ShardView T,
                                                     u64 *__restrict__ resp, u32 *__restrict__ runlen)
{
    for (u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x; p < nq; p += (u64)gridDim.x * blockDim.x) {
        u32 run;
        resp[p] = answer_one(T, queries, p, exact, run);
        runlen[p] = run;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) runlen[nq] = 0;     // sentinel: off[nq] = total after the scan
}

// The mailbox form, one launch per source: the finished answer word goes straight into the source's mailbox
// (`resp` is PEER memory: coalesced 8-byte stores over NVLink), the entry runs into a local stream in chunks a warp
// reserves with one atomic (no scan, no second pass; the answers carry explicit offsets, so the unused tail of a chunk
// may stay a hole); the stream is copied to the source afterwards.
__global__ void __launch_bounds__(256) answer_fused_kernel(const u64 *__restrict__ queries, u64 nq, int exact, const __grid_constant__ ShardView T,
                                                           u64 *__restrict__ resp, u32 *__restrict__ ent_out, u64 ecap,
                                                           unsigned long long *__restrict__ cursor)
{
    const int lane = threadIdx.x & 31;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    unsigned long long wbase = 0;
    u32 wleft = 0;
    for (u64 p0 = (u64)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); p0 < nq; p0 += stride) {      // warp-uniform trip count
        const u64 p = p0 + lane;
        u32 run = 0;
        u64 answer = 0;
        if (p < nq) answer = answer_one(T, queries, p, exact, run);
        u32 incl = run;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const u32 y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
        const u32 total = __shfl_sync(0xffffffffu, incl, 31);
        if (total > wleft) {          // a fresh chunk of the stream for this warp (what is left of the old one stays a hole)
            const u32 take = total > kEntryChunk ? total : kEntryChunk;
            if (lane == 31) wbase = atomicAdd(cursor, (unsigned long long)take);
            wbase = __shfl_sync(0xffffffffu, wbase, 31);
            wleft = take;
        }
        const unsigned long long base = wbase;
        wbase += total; wleft -= total;
        if (run) {
            const u64 at = base + incl - run;
            if (at + run <= ecap) {                       // (an overflow is reported by the host from the cursor)
                const u32 *src = T.entries + slot_get_payload(answer);
                for (u32 e = 0; e < run; ++e) ent_out[at + e] = src[e];
            }
            answer = answer_encode(run, at);
        }
        if (p < nq) resp[p] = answer;
    }
}

// entry runs -> the stream of the query's source, answer payload := offset inside that stream
__global__ void __launch_bounds__(256) answer_runs_kernel(u64 *__restrict__ resp, const u32 *__restrict__ runlen, const u32 *__restrict__ off, u64 nq,
                                                          const u64 *__restrict__ seg_start /*[world+1]*/, int world,
                                                          const u32 *__restrict__ entries, u32 *__restrict__ out)
{
    for (u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x; p < nq; p += (u64)gridDim.x * blockDim.x) {
        const u32 c = runlen[p];
        if (c == 0) continue;
        int s = 0;
        while (s + 1 < world && seg_start[s + 1] <= p) ++s;
        const u32 rel = off[p] - off[seg_start[s]];
        const u64 src = slot_get_payload(resp[p]);
        for (u32 e = 0; e < c; ++e) out[off[p] + e] = entries[src + e];
        resp[p] = answer_encode(c, rel);
    }
}

__global__ void seg_totals_kernel(const u32 *__restrict__ off, const u64 *__restrict__ seg_start, int world, u64 *__restrict__ out)
{
    const int s = threadIdx.x;
    if (s < world) out[s] = (u64)(off[seg_start[s + 1]] - off[seg_start[s]]);
}

// ---- source: answers -> wslot ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) route_finish_kernel(const u64 *__restrict__ resp, const u32 *__restrict__ qmap, u64 Q,
                                                           const u64 *__restrict__ qbase /*[world+1]*/, const u64 *__restrict__ ebase /*[world]*/,
                                                           int world, u64 *__restrict__ wslot)
{
    for (u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x; p < Q; p += (u64)gridDim.x * blockDim.x) {
        u64 w = resp[p];
        const u32 c = slot_get_count(w);
        if (c >= 2 && c < (u32)kHashThreshold) {
            int g = 0;
            while (g + 1 < world && qbase[g + 1] <= p) ++g;
            w += ebase[g];
        }
        wslot[qmap[p]] = w;
    }
}

// ---- id lists ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) flag_equal_kernel(const uint8_t *__restrict__ a, u64 n, uint8_t value, u32 *__restrict__ flag)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) flag[i] = a[i] == value;
}
__global__ void __launch_bounds__(256) compact_list_kernel(const u32 *__restrict__ flag, const u32 *__restrict__ idx, u64 n, u32 base, u32 *__restrict__ out)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        if (flag[i]) out[idx[i]] = base + (u32)i;
}

static ShardView shard_view(const Context &c)
{
    ShardView T;
    T.slots = c.slots.p; T.nsec = c.cap / kSlotsPerSector; T.entries = c.entries.p; T.F = c.F.p; T.RC = c.RC.p; T.len = c.len.p;
    T.SW = c.SW; T.SWS = c.SWS; T.h = c.h;
    return T;
}

static unsigned sm_grid(u64 n, unsigned per_block, unsigned blocks_per_sm)
{
    u64 g = (n + per_block - 1) / per_block;
    const u64 cap = (u64)kSMs * blocks_per_sm;
    if (g > cap) g = cap;
    return g ? (unsigned)g : 1u;
}

// ascending list of base + i for the i in [0, n) with a[i] == value -> c.rt_ids; returns its length
static u64 build_id_list(Context &c, const uint8_t *a, u64 n, uint8_t value, u32 base)
{
    cudaStream_t st = c.stream;
    if (n == 0) { c.rt_ids.alloc(0, st); return 0; }
    DevBuf<u32> flag(n, st), idx(n, st), d_total(1, st);
    flag_equal_kernel<<<sm_grid(n, 1024, 8), 256, 0, st>>>(a, n, value, flag.p);
    SG_LAUNCHED();
    exclusive_scan_u32(flag.p, idx.p, n, d_total.p, st);
    u32 cnt = 0;
    SG_CUDA(cudaMemcpyAsync(&cnt, d_total.p, sizeof(u32), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    c.rt_ids.alloc(cnt, st);
    if (cnt) {
        compact_list_kernel<<<sm_grid(n, 1024, 8), 256, 0, st>>>(flag.p, idx.p, n, base, c.rt_ids.p);
        SG_LAUNCHED();
    }
    return cnt;
}

// what = 0: reads [first, first + count) (0-based indices);  1: the reads in state 0 after phase B (phase C);
//        2: the reads of this rank's phase-A slice flagged for the redo pass.
static void select_batch(Context &c, int what, u64 first, u64 count, int exact, int world)
{
    SG_CHECK(c.have_reads, "organize_reads must run first");
    SG_CHECK(world >= 1 && world <= kMaxWorld, "bad world size");
    SG_CHECK(what >= 0 && what <= 2, "bad batch kind");
    const u64 U = c.cnt.unique_reads;
    c.rt_state = 0; c.rt_for_c = false;
    c.rt_what = what; c.rt_exact = exact != 0; c.rt_world = world;
    c.rt_is_list = what != 0;
    if (what == 0) {
        SG_CHECK(first <= U && count <= U - first, "batch outside the reads");
        SG_CHECK(count == 0 || (first >= c.pa_lo && first + count <= c.pa_hi), "batch outside this rank's phase-A slice");
        c.rt_first = first; c.rt_n = count;
    } else if (what == 1) {
        SG_CHECK(c.have_phase_b, "phase B must run before the phase-C reads are routed");
        SG_CHECK(exact, "phase C needs verified probes");
        c.rt_first = 0; c.rt_n = build_id_list(c, c.explored.p, U, 0, 0);
    } else {
        SG_CHECK(exact, "the redo pass needs verified probes");
        c.rt_first = 0; c.rt_n = build_id_list(c, c.rt_redo.p, c.pa_hi - c.pa_lo, 1, (u32)c.pa_lo);
    }
    const int wstride = c.max_len - c.h + 1 > 1 ? c.max_len - c.h + 1 : 1;
    c.rt_wstride = (u32)wstride;
    SG_CHECK(c.rt_n * (u64)wstride < 0xFFFFFFFFull, "routed batch too large: at most 2^32 windows per batch");
    for (int g = 0; g < kMaxWorld; ++g) c.rt_counts[g] = 0;
    c.rt_Q = 0;
}

void stage_route_begin(Context &c, int what, u64 first, u64 count, int exact, int world, void **queries, u64 *counts)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    select_batch(c, what, first, count, exact, world);
    const u64 n = c.rt_n;
    const int wstride = (int)c.rt_wstride;
    c.rt_mailbox = false;
    if (n > 0) {
        DevBuf<unsigned long long> d_cnt(world, st);
        SG_CUDA(cudaMemsetAsync(d_cnt.p, 0, world * sizeof(unsigned long long), st));
        const u32 *ids = c.rt_is_list ? c.rt_ids.p : nullptr;
        const unsigned grid = sm_grid(n, RT_WARPS, 8);
        RouteDst D = {};
        route_kernel<false><<<grid, RT_WARPS * 32, 0, st>>>(c.F.p, c.SW, c.SWS, c.h, ids, c.rt_first, n, c.rt_wstride, world, exact, d_cnt.p, D, nullptr);
        SG_LAUNCHED();
        unsigned long long h_cnt[kMaxWorld];
        u64 h_base[kMaxWorld];
        SG_CUDA(cudaMemcpyAsync(h_cnt, d_cnt.p, world * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        SG_CUDA(cudaStreamSynchronize(st));
        u64 Q = 0;
        for (int g = 0; g < world; ++g) { h_base[g] = Q; c.rt_counts[g] = h_cnt[g]; Q += h_cnt[g]; }
        c.rt_Q = Q;
        c.rt_queries.alloc(Q * (exact ? 2 : 1), st);
        c.rt_qmap.alloc(Q, st);
        c.rt_wslot.alloc(n * (u64)wstride, st);
        SG_CUDA(cudaMemsetAsync(d_cnt.p, 0, world * sizeof(unsigned long long), st));
        for (int g = 0; g < world; ++g) { D.dst[g] = c.rt_queries.p + h_base[g] * (exact ? 2 : 1); D.qoff[g] = h_base[g]; }
        route_kernel<true><<<grid, RT_WARPS * 32, 0, st>>>(c.F.p, c.SW, c.SWS, c.h, ids, c.rt_first, n, c.rt_wstride, world, exact, d_cnt.p, D, c.rt_qmap.p);
        SG_LAUNCHED();
        SG_CUDA(cudaStreamSynchronize(st));      // the caller reads the queries from another stream
    }
    if (queries) *queries = c.rt_Q ? (void *)c.rt_queries.p : nullptr;
    if (counts) for (int g = 0; g < world; ++g) counts[g] = c.rt_counts[g];
    c.rt_state = 1;
}

// Owner side.  `queries` (device): the streams received from source 0, 1, .. world-1 back to back,
// counts_per_source[s] queries each.  Answers in the same order; entry stream of source s = entry_counts[s] words.
__global__ void __launch_bounds__(256) sum_runlen_kernel(const u32 *__restrict__ v, u64 n, unsigned long long *__restrict__ out)
{
    unsigned long long acc = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) acc += v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

void stage_shard_answer(Context &c, const void *queries, const u64 *counts_per_source, int exact, int world, void **responses, void **entries,
                        u64 *entry_counts)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    SG_CHECK(c.have_table, "build_hash_table[_shard] must run first");
    SG_CHECK(world == c.tb_world, "world size differs from the one the table shard was built for");
    u64 nq = 0;
    u64 h_seg[kMaxWorld + 1];
    for (int s = 0; s < world; ++s) { h_seg[s] = nq; nq += counts_per_source[s]; }
    h_seg[world] = nq;
    for (int s = 0; s < world; ++s) entry_counts[s] = 0;
    *responses = nullptr; *entries = nullptr;
    if (nq == 0) return;
    SG_CHECK(queries != nullptr, "null query buffer");
    c.an_resp.alloc(nq, st);
    DevBuf<u32> runlen(nq + 1, st), off(nq + 1, st), d_total(1, st);
    DevBuf<u64> d_seg(world + 1, st), d_ecnt(world, st);
    SG_CUDA(cudaMemcpyAsync(d_seg.p, h_seg, (world + 1) * sizeof(u64), cudaMemcpyHostToDevice, st));
    const ShardView T = shard_view(c);
    answer_kernel<<<sm_grid(nq, 256, 8), 256, 0, st>>>((const u64 *)queries, nq, exact, T, c.an_resp.p, runlen.p);
    SG_LAUNCHED();
    // up to 99 entries per query: the grand total is checked in 64 bits before the 32-bit scan is trusted
    DevBuf<unsigned long long> d_t64(1, st);
    SG_CUDA(cudaMemsetAsync(d_t64.p, 0, sizeof(unsigned long long), st));
    sum_runlen_kernel<<<sm_grid(nq, 256, 8), 256, 0, st>>>(runlen.p, nq, d_t64.p);
    SG_LAUNCHED();
    exclusive_scan_u32(runlen.p, off.p, nq + 1, d_total.p, st);
    seg_totals_kernel<<<1, kMaxWorld, 0, st>>>(off.p, d_seg.p, world, d_ecnt.p);
    SG_LAUNCHED();
    u32 total = 0;
    u64 h_ecnt[kMaxWorld];
    unsigned long long total64 = 0;
    SG_CUDA(cudaMemcpyAsync(&total64, d_t64.p, sizeof(total64), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaMemcpyAsync(&total, d_total.p, sizeof(u32), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaMemcpyAsync(h_ecnt, d_ecnt.p, world * sizeof(u64), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    SG_CHECK(total64 < 0xFFFFFFFFull, "more than 2^32 bucket entries in one routed batch: use smaller batches");
    c.an_entries.alloc(total, st);
    if (total) {
        answer_runs_kernel<<<sm_grid(nq, 256, 8), 256, 0, st>>>(c.an_resp.p, runlen.p, off.p, nq, d_seg.p, world, c.entries.p, c.an_entries.p);
        SG_LAUNCHED();
    }
    SG_CUDA(cudaStreamSynchronize(st));
    for (int s = 0; s < world; ++s) entry_counts[s] = h_ecnt[s];
    *responses = c.an_resp.p;
    *entries = total ? (void *)c.an_entries.p : nullptr;
}

// Source side.  `responses`: one word per query in the order of route_begin's streams; `entries`: the entry
// streams of owner 0, 1, .. back to back (entry_counts[g] words each).  Both device pointers.
void stage_route_finish(Context &c, const void *responses, const void *entries, const u64 *entry_counts)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    SG_CHECK(c.rt_state == 1, "route_begin must precede route_finish");
    const int world = c.rt_world;
    u64 h_qbase[kMaxWorld + 1], h_ebase[kMaxWorld], E = 0, Q = 0;
    for (int g = 0; g < world; ++g) { h_qbase[g] = Q; Q += c.rt_counts[g]; h_ebase[g] = E; E += entry_counts[g]; }
    h_qbase[world] = Q;
    SG_CHECK(E < (1ull << 32), "entry streams too long for one batch");
    c.rt_wentries.alloc(E, st);
    if (E) SG_CUDA(cudaMemcpyAsync(c.rt_wentries.p, entries, E * sizeof(u32), cudaMemcpyDeviceToDevice, st));
    if (Q) {
        SG_CHECK(responses != nullptr, "null answer buffer");
        DevBuf<u64> d_qbase(world + 1, st), d_ebase(world, st);
        SG_CUDA(cudaMemcpyAsync(d_qbase.p, h_qbase, (world + 1) * sizeof(u64), cudaMemcpyHostToDevice, st));
        SG_CUDA(cudaMemcpyAsync(d_ebase.p, h_ebase, world * sizeof(u64), cudaMemcpyHostToDevice, st));
        route_finish_kernel<<<sm_grid(Q, 1024, 8), 256, 0, st>>>((const u64 *)responses, c.rt_qmap.p, Q, d_qbase.p, d_ebase.p, world, c.rt_wslot.p);
        SG_LAUNCHED();
    }
    SG_CUDA(cudaStreamSynchronize(st));       // the caller's buffers may be reused on return
    c.rt_entries_view = c.rt_wentries.p;
    c.rt_state = 2;
    c.rt_for_c = c.rt_what == 1;
}


// =====================================================================================================================
// The same exchange over PEER MEMORY (NVLink / NVSwitch P2P) instead of NCCL.  Every rank owns one "mailbox" (one
// cudaMalloc block, opened by the other ranks through CUDA IPC, or plain pointers inside one process):
//
//   counts   [world]            u64   queries source s sent me in this batch
//   flags    [world]            u64   barrier epochs: peer r has arrived at barrier number flags[r]
//   queries  [world][cap][2]    u64   stream of source s (key hashes, or 128-bit keys)      -- I answer these as OWNER
//   answers  [world][cap]       u64   answers of owner g to the queries I sent it           -- I consume these as SOURCE
//   entries  [world][ecap]      u32   entry stream of owner g for my queries
//
// route_post    the routing kernel stores every query straight into its owner's mailbox (the all-to-all "dispatch" is
//               the kernel's own store traffic, tile by tile) and publishes the counts;   [barrier between the ranks]
// answer_post   the owner answers out of its mailbox and copies answers + entries into the sources' mailboxes over
//               NVLink ("combine");                                                     [barrier between the ranks]
// route_collect the source scatters the answers from its own mailbox into wslot; the search kernel reads the entry
//               streams in place.  Segments have a fixed capacity, so no sizes travel ahead of the data.
// =====================================================================================================================
static size_t mb_align(size_t x) { return (x + 255) & ~(size_t)255; }
static size_t mb_off_counts() { return 0; }
static size_t mb_off_flags(int world) { return mb_align((size_t)world * 8); }                // barrier epochs, one per peer
static size_t mb_off_queries(int world) { return mb_off_flags(world) + mb_align((size_t)world * 8); }
static size_t mb_off_answers(int world, u64 cap) { return mb_off_queries(world) + mb_align((size_t)world * cap * 16); }
static size_t mb_off_entries(int world, u64 cap) { return mb_off_answers(world, cap) + mb_align((size_t)world * cap * 8); }
static size_t mb_bytes(int world, u64 cap, u64 ecap) { return mb_off_entries(world, cap) + mb_align((size_t)world * ecap * 4); }

void stage_mailbox_create(Context &c, int rank, int world, u64 cap_windows, void *ipc_handle_out, void **local_ptr)
{
    SG_CHECK(world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world, "bad rank / world");
    SG_CHECK(cap_windows >= 1 && cap_windows < 0xFFFFFFFFull && (u64)world * cap_windows < (1ull << 33), "bad mailbox capacity");
    stage_mailbox_destroy(c);
    Mailbox &m = c.mb;
    // entry segments: room for `factor` bucket entries per window on average (entries travel only for buckets of 2..99
    // reads: 0.25 per window at cfg2, < 0.1 at cfg4; SAGE2GPU_MAILBOX_ENTRY_FACTOR raises it for repeat-rich or very deep
    // data) + the holes the chunked reservation of answer_fused_kernel can leave.  This is NOT a worst case (a bucket holds
    // up to 99 entries): a batch that needs more fails loudly ("entry stream exceeds the mailbox capacity") and the
    // caller reruns with a larger factor, smaller batches or the NCCL transport, which sizes its buffers exactly.
    static const u64 efactor = [] { const char *e = getenv("SAGE2GPU_MAILBOX_ENTRY_FACTOR"); const long v = e ? atol(e) : 2; return (u64)(v < 1 ? 1 : v); }();
    m.world = world; m.rank = rank; m.cap = cap_windows; m.ecap = efactor * cap_windows + (u64)kSMs * 8 * 8 * kEntryChunk;
    SG_CHECK((u64)world * m.ecap < (1ull << 33), "mailbox too large for the 33-bit answer payload");
    m.bytes = mb_bytes(world, m.cap, m.ecap);
    SG_CUDA(cudaMalloc((void **)&m.base, m.bytes));          // plain cudaMalloc: pool memory cannot be exported through IPC
    SG_CUDA(cudaMemset(m.base, 0, mb_off_queries(world)));
    for (int r = 0; r < kMaxWorld; ++r) { m.peer[r] = nullptr; m.ipc[r] = false; }
    m.peer[rank] = m.base;
    if (ipc_handle_out) {
        cudaIpcMemHandle_t hnd;
        SG_CUDA(cudaIpcGetMemHandle(&hnd, m.base));
        static_assert(sizeof(hnd) == 64, "CUDA IPC handles are 64 bytes");
        memcpy(ipc_handle_out, &hnd, sizeof(hnd));
    }
    if (local_ptr) *local_ptr = m.base;
}

// the mailbox of `peer_rank`: an IPC handle exported by another process, or (same process) its pointer
void stage_mailbox_open(Context &c, int peer_rank, const void *ipc_handle, void *ptr)
{
    Mailbox &m = c.mb;
    SG_CHECK(m.base != nullptr, "mailbox_create must run first");
    SG_CHECK(peer_rank >= 0 && peer_rank < m.world, "bad peer rank");
    if (peer_rank == m.rank) return;
    if (ipc_handle) {
        cudaIpcMemHandle_t hnd;
        memcpy(&hnd, ipc_handle, sizeof(hnd));
        void *p = nullptr;
        SG_CUDA(cudaIpcOpenMemHandle(&p, hnd, cudaIpcMemLazyEnablePeerAccess));
        m.peer[peer_rank] = (char *)p; m.ipc[peer_rank] = true;
    } else {
        SG_CHECK(ptr != nullptr, "null peer pointer");
        // a mailbox on another GPU of this process: the routing and barrier kernels store into it, which needs peer access
        cudaPointerAttributes a;
        SG_CUDA(cudaPointerGetAttributes(&a, ptr));
        if (a.type == cudaMemoryTypeDevice && a.device != c.device) {
            int can = 0;
            SG_CUDA(cudaDeviceCanAccessPeer(&can, c.device, a.device));
            SG_CHECK(can, "GPU " + std::to_string(c.device) + " cannot access the memory of GPU " + std::to_string(a.device) +
                              " (no peer access between them): the mailbox of rank " + std::to_string(peer_rank) + " cannot be used");
            const cudaError_t e = cudaDeviceEnablePeerAccess(a.device, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else SG_CUDA(e);
        }
        m.peer[peer_rank] = (char *)ptr; m.ipc[peer_rank] = false;
    }
}

void stage_mailbox_destroy(Context &c)
{
    Mailbox &m = c.mb;
    if (!m.base) return;
    cudaStreamSynchronize(c.stream);
    for (int r = 0; r < m.world; ++r) if (r != m.rank && m.peer[r] && m.ipc[r]) cudaIpcCloseMemHandle(m.peer[r]);
    cudaFree(m.base);
    m = Mailbox();
}

__global__ void publish_counts_kernel(const unsigned long long *__restrict__ cnt, const __grid_constant__ RouteDst D, int world)
{
    const int g = threadIdx.x;
    if (g < world) *D.dst[g] = cnt[g];        // counts[rank] in owner g's mailbox
}

// Barrier between the ranks ON THE DEVICE: one thread per peer stores this rank's epoch into the peer's mailbox (after a
// system-scope fence: everything this rank stored into peer memory before is visible first) and then waits until the
// peer's epoch has arrived here.  Stream-ordered, no host round trip through a collective.  A peer that never arrives
// (a dead rank) ends the wait after 60 s (SAGE2GPU_BARRIER_TIMEOUT_S) with an error instead of hanging the GPU; the
// mailbox is released then, because the ranks' epochs no longer agree.
__global__ void mailbox_barrier_kernel(const __grid_constant__ RouteDst D /* dst[g] = flags[rank] in peer g's mailbox */,
                                       const volatile u64 *__restrict__ my_flags, u64 epoch, int world, int rank, long long timeout_clocks,
                                       u32 *__restrict__ timed_out)
{
    const int g = threadIdx.x;
    if (g >= world || g == rank) return;
    __threadfence_system();
    *reinterpret_cast<volatile u64 *>(D.dst[g]) = epoch;
    const long long t0 = clock64();
    while (my_flags[g] < epoch) {
        __nanosleep(200);
        if (clock64() - t0 > timeout_clocks) { *timed_out = 1; break; }
    }
    __threadfence_system();
}

void stage_mailbox_barrier(Context &c)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    Mailbox &m = c.mb;
    SG_CHECK(m.base != nullptr, "mailbox_create must run first");
    if (m.world == 1) return;
    RouteDst D = {};
    for (int g = 0; g < m.world; ++g) {
        SG_CHECK(m.peer[g] != nullptr, "a peer mailbox has not been opened");
        D.dst[g] = (u64 *)(m.peer[g] + mb_off_flags(m.world)) + m.rank;
    }
    DevBuf<u32> d_to(1, st);
    SG_CUDA(cudaMemsetAsync(d_to.p, 0, sizeof(u32), st));
    ++m.epoch;
    // a peer may be late by seconds (lazy module load, allocator stalls, uneven batches): 60 s by default
    // (SAGE2GPU_BARRIER_TIMEOUT_S), counted in SM clocks at ~2 GHz
    static const long long timeout_clocks = [] { const char *e = getenv("SAGE2GPU_BARRIER_TIMEOUT_S"); const long v = e ? atol(e) : 60; return (long long)(v < 1 ? 1 : v) * 2000000000ll; }();
    mailbox_barrier_kernel<<<1, kMaxWorld, 0, st>>>(D, (const volatile u64 *)(m.base + mb_off_flags(m.world)), m.epoch, m.world, m.rank, timeout_clocks, d_to.p);
    SG_LAUNCHED();
    u32 h_to = 0;
    SG_CUDA(cudaMemcpyAsync(&h_to, d_to.p, sizeof(u32), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    if (h_to != 0) {
        // this rank has already published its epoch, so the peers pass this barrier: the mailbox is unusable from here on
        // (the epochs of the ranks no longer agree).  Drop it; the next build has to create and open the mailboxes again.
        stage_mailbox_destroy(c);
        throw CudaError("mailbox barrier timed out: a peer rank never arrived (mailbox released; create it again)");
    }
}

void stage_route_post(Context &c, int what, u64 first, u64 count, int exact, u64 *n_reads)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    Mailbox &m = c.mb;
    SG_CHECK(m.base != nullptr, "mailbox_create must run first");
    const int world = m.world, rank = m.rank;
    for (int g = 0; g < world; ++g) SG_CHECK(m.peer[g] != nullptr, "a peer mailbox has not been opened");
    select_batch(c, what, first, count, exact, world);
    c.rt_mailbox = true;
    const u64 n = c.rt_n;
    SG_CHECK(n * (u64)c.rt_wstride <= m.cap, "routed batch larger than the mailbox capacity");
    if (n_reads) *n_reads = n;
    DevBuf<unsigned long long> d_cnt(world, st);
    SG_CUDA(cudaMemsetAsync(d_cnt.p, 0, world * sizeof(unsigned long long), st));
    RouteDst D = {}, C = {};
    for (int g = 0; g < world; ++g) {
        D.dst[g] = (u64 *)(m.peer[g] + mb_off_queries(world)) + (u64)rank * m.cap * 2;      // my segment in owner g's mailbox
        D.qoff[g] = (u64)g * m.cap;
        C.dst[g] = (u64 *)(m.peer[g] + mb_off_counts()) + rank;
    }
    if (n > 0) {
        c.rt_qmap.alloc((u64)world * m.cap, st);
        c.rt_wslot.alloc(n * (u64)c.rt_wstride, st);
        const u32 *ids = c.rt_is_list ? c.rt_ids.p : nullptr;
        route_kernel<true><<<sm_grid(n, RT_WARPS, 8), RT_WARPS * 32, 0, st>>>(c.F.p, c.SW, c.SWS, c.h, ids, c.rt_first, n, c.rt_wstride, world, exact,
                                                                            d_cnt.p, D, c.rt_qmap.p);
        SG_LAUNCHED();
    }
    publish_counts_kernel<<<1, kMaxWorld, 0, st>>>(d_cnt.p, C, world);
    SG_LAUNCHED();
    unsigned long long h_cnt[kMaxWorld];
    SG_CUDA(cudaMemcpyAsync(h_cnt, d_cnt.p, world * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));       // every store to the peers has landed when the caller enters the barrier
    u64 Q = 0;
    for (int g = 0; g < world; ++g) { c.rt_counts[g] = h_cnt[g]; Q += h_cnt[g]; }
    c.rt_Q = Q;
    c.rt_state = 1;
}

// owner: answer what the sources posted (after the barrier that follows route_post on every rank)
void stage_answer_post(Context &c, int exact, u64 *bytes_sent)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    Mailbox &m = c.mb;
    SG_CHECK(m.base != nullptr, "mailbox_create must run first");
    SG_CHECK(c.have_table, "build_hash_table[_shard] must run first");
    const int world = m.world, rank = m.rank;
    SG_CHECK(world == c.tb_world && rank == c.tb_rank, "the mailbox and the table shard disagree about rank / world");
    u64 h_cnt[kMaxWorld], nq = 0;
    SG_CUDA(cudaMemcpyAsync(h_cnt, m.base + mb_off_counts(), world * sizeof(u64), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    for (int s = 0; s < world; ++s) { SG_CHECK(h_cnt[s] <= m.cap, "posted count exceeds the mailbox capacity"); nq += h_cnt[s]; }
    if (bytes_sent) *bytes_sent = 0;
    if (nq == 0) return;
    SG_CHECK(nq < 0xFFFFFFFFull, "too many queries for one batch");
    // one fused launch per source: answers land in the source's mailbox while the kernel runs ("combine")
    const ShardView T = shard_view(c);
    DevBuf<unsigned long long> d_cur(world, st);
    SG_CUDA(cudaMemsetAsync(d_cur.p, 0, world * sizeof(unsigned long long), st));
    c.an_entries.alloc((u64)world * m.ecap, st);
    const u64 *qin = (const u64 *)(m.base + mb_off_queries(world));
    for (int s = 0; s < world; ++s) {
        if (h_cnt[s] == 0) continue;
        u64 *ans = (u64 *)(m.peer[s] + mb_off_answers(world, m.cap)) + (u64)rank * m.cap;
        answer_fused_kernel<<<sm_grid(h_cnt[s], 256, 8), 256, 0, st>>>(qin + (u64)s * m.cap * 2, h_cnt[s], exact, T, ans, c.an_entries.p + (u64)s * m.ecap,
                                                                         m.ecap, d_cur.p + s);
        SG_LAUNCHED();
    }
    unsigned long long h_ecnt[kMaxWorld];
    SG_CUDA(cudaMemcpyAsync(h_ecnt, d_cur.p, world * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    u64 sent = 0;
    for (int s = 0; s < world; ++s) {
        SG_CHECK(h_ecnt[s] <= m.ecap, "entry stream exceeds the mailbox capacity");
        if (h_ecnt[s]) {
            u32 *ent = (u32 *)(m.peer[s] + mb_off_entries(world, m.cap)) + (u64)rank * m.ecap;
            SG_CUDA(cudaMemcpyAsync(ent, c.an_entries.p + (u64)s * m.ecap, h_ecnt[s] * sizeof(u32), cudaMemcpyDeviceToDevice, st));
        }
        if (s != rank) sent += h_cnt[s] * 8 + h_ecnt[s] * 4;
    }
    SG_CUDA(cudaStreamSynchronize(st));
    if (bytes_sent) *bytes_sent = sent;
}

__global__ void __launch_bounds__(256) route_collect_kernel(const u64 *__restrict__ answers, const u32 *__restrict__ qmap, u64 cap, u64 ecap,
                                                            const __grid_constant__ RouteDst N /* qoff[g] = my queries to owner g */, int world,
                                                            u64 *__restrict__ wslot)
{
    for (int g = 0; g < world; ++g) {
        const u64 cnt = N.qoff[g];
        const u64 *a = answers + (u64)g * cap;
        const u32 *qm = qmap + (u64)g * cap;
        for (u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x; p < cnt; p += (u64)gridDim.x * blockDim.x) {
            u64 w = a[p];
            const u32 c = slot_get_count(w);
            if (c >= 2 && c < (u32)kHashThreshold) w += (u64)g * ecap;
            wslot[qm[p]] = w;
        }
    }
}

// source: after the barrier that follows answer_post on every rank
void stage_route_collect(Context &c)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    Mailbox &m = c.mb;
    SG_CHECK(c.rt_state == 1 && c.rt_mailbox, "route_post must precede route_collect");
    const int world = m.world;
    if (c.rt_Q) {
        RouteDst N = {};
        for (int g = 0; g < world; ++g) N.qoff[g] = c.rt_counts[g];
        route_collect_kernel<<<sm_grid(c.rt_Q, 1024, 8), 256, 0, st>>>((const u64 *)(m.base + mb_off_answers(world, m.cap)), c.rt_qmap.p, m.cap, m.ecap, N,
                                                                       world, c.rt_wslot.p);
        SG_LAUNCHED();
        SG_CUDA(cudaStreamSynchronize(st));
    }
    c.rt_entries_view = (const u32 *)(m.base + mb_off_entries(world, m.cap));
    c.rt_state = 2;
    c.rt_for_c = c.rt_what == 1;
}

}  // namespace sg
