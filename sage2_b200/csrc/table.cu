// table.cu -- step 2 on device: the prefix/suffix table (K3).  Restates
// HashTable::hashPrefixesAndSuffix / hashTableInsert (economyGraph/hashTable.cpp:70-188).
//
// Observable semantics kept exactly: key (h = min(k,64) bases) -> all (readId,type) sharing it, in
// (readId asc, type asc) order; a key with >= 100 entries is invisible to searches.  Layout:
//   slots[cap]   : open-addressing index, one 64-bit slot per DISTINCT key, grouped in 32-byte sectors
//                  of 4 (a probe reads one sector), filled with 64-bit atomicCAS:
//                  tag | min(count,127) | payload (core.cuh).  payload = the key's only entry
//                  (count == 1), a representative entry (count >= 100, masked) or the offset of the
//                  key's run in entries[] (2 <= count <= 99).
//   entries[M]   : (readId0<<2 | type) of every key with 2..99 entries, each run sorted ascending, which
//                  is the reference's bucket order (insertion order, hashTable.cpp:94-109).
// Like the reference (hashTable.cpp:150-160) a slot does not store its 128-bit key: a tag match is
// confirmed by re-extracting the key from the read of the slot's representative entry.
//
// Four passes over the 4U entries:
//   1 insert  : find-or-claim the key's slot (atomicCAS on an empty slot, saturating CAS increment of
//               the count on a match), remember the slot per entry
//   2 offsets : exclusive scan of the 2..99 counts over the slot array, rewrite those slots' payload
//   3 fill    : every entry of such a key takes the next position of its run (atomic cursor)
//   4 order   : insertion sort of every run (< 100 entries)
// When the slot index is much larger than L2 (cfg4: 1.3 GB) passes 1 and 3 are random accesses that cost a 128-byte
// line of HBM traffic each (ncu: 252 bytes per inserted entry).  Then the entries are first bucketed by the top 8 bits
// of their key hash -- home_sector() is monotone in the hash, so a bucket is one 1/256 range of the slot array -- with
// ONE radix pass over (hash, entry) records, and passes 1 and 3 walk the records in that order: the slots they touch
// are L2-resident while their bucket is being worked on, every line of the index is fetched once.
#include <stdlib.h>
#include "context.h"

namespace sg {

constexpr u64 kCountOne = 1ull << 33;
constexpr u32 kNotOwned = 0xFFFFFFFFu;      // where[] of an entry whose key belongs to another shard

__device__ __forceinline__ u64 load_slot(const u64 *p) { return *reinterpret_cast<const volatile u64 *>(p); }

__global__ void __launch_bounds__(256) table_insert_kernel(const u64 *__restrict__ F, const u64 *__restrict__ RC,
                                                            const uint16_t *__restrict__ len, u64 U, int SW, int SWS, int h,
                                                            u64 *__restrict__ slots, u64 nsec, u32 *__restrict__ where,
                                                            int rank, int world, u32 *__restrict__ overflow)
{
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < 4 * U; t += (u64)gridDim.x * blockDim.x) {
        const u64 rid = t >> 2;
        const int type = (int)(t & 3);
        u64 v0, v1;
        entry_key(F + rid * SWS, RC + rid * SWS, SW, len[rid], h, type, v0, v1);
        const u64 hsh = hash_key(v0, v1);
        if (key_owner(hsh, world) != rank) { where[t] = kNotOwned; continue; }      // another shard's key
        const u64 tag = slot_tag(hsh);
        u64 sec = home_sector(hsh, nsec);
        bool done = false;
        u64 tries = 0;
        while (!done) {
            for (int q = 0; q < kSlotsPerSector && !done; ++q) {
                u64 *sp = slots + kSlotsPerSector * sec + q;
                u64 cur = load_slot(sp);
                if (cur == 0) {
                    const u64 old = atomicCAS((unsigned long long *)sp, 0ull, (unsigned long long)slot_encode(hsh, 1, t));
                    if (old == 0) { where[t] = (u32)(kSlotsPerSector * sec + q); done = true; break; }
                    cur = old;
                }
                if (slot_get_tag(cur) != tag) continue;
                // same tag: same key?  (the representative entry never changes once the slot is claimed)
                const u32 rep = (u32)slot_get_payload(cur);
                const u64 r2 = rep >> 2;
                u64 w0, w1;
                entry_key(F + r2 * SWS, RC + r2 * SWS, SW, len[r2], h, (int)(rep & 3), w0, w1);
                if (w0 != v0 || w1 != v1) continue;
                while (slot_get_count(cur) < 127) {            // saturating: >= 100 is all a search needs to know
                    const u64 old = atomicCAS((unsigned long long *)sp, (unsigned long long)cur, (unsigned long long)(cur + kCountOne));
                    if (old == cur) break;
                    cur = old;
                }
                where[t] = (u32)(kSlotsPerSector * sec + q);
                done = true;
            }
            sec = (sec + 1 == nsec) ? 0 : sec + 1;
            if (++tries > nsec) { *overflow = 1; where[t] = kNotOwned; break; }      // index full: reported, never silent
        }
    }
}

// ---- bucketed build: (hash, entry) records of the keys this shard owns ---------------------------------------------------
// A record carries what decides key equality, so that the build never goes back to the reads: hash_key() is a bijection
// of v1 for a fixed v0 (mix64 is invertible), hence two keys are equal iff their hashes and their v0 words are.  For
// h <= 32, v0 is always 0 and the hash alone decides; otherwise v0 travels in a column B of its own.
// one thread per read: its four keys.  world <= 1: record 4 rid + type sits at its own index; else the owned records are
// compacted (one atomicAdd per block and round)
__global__ void __launch_bounds__(256) table_keys_kernel(const u64 *__restrict__ F, const u64 *__restrict__ RC, const uint16_t *__restrict__ len,
                                                          u64 U, int SW, int SWS, int h, int rank, int world,
                                                          u64 *__restrict__ A, u64 *__restrict__ B, u32 *__restrict__ V, u64 room,
                                                          unsigned long long *__restrict__ n_out)
{
    __shared__ u32 s_warp[8];
    __shared__ unsigned long long s_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (u64 r0 = (u64)blockIdx.x * 256; r0 < U; r0 += (u64)gridDim.x * 256) {
        const u64 rid = r0 + threadIdx.x;
        u64 hs[4] = { 0, 0, 0, 0 }, ks[4] = { 0, 0, 0, 0 };
        u32 own = 0;
        if (rid < U) {
            const int l = len[rid];
#pragma unroll
            for (int type = 0; type < 4; ++type) {
                u64 v1;
                entry_key(F + rid * SWS, RC + rid * SWS, SW, l, h, type, ks[type], v1);
                hs[type] = hash_key(ks[type], v1);
                if (world <= 1 || key_owner(hs[type], world) == rank) own |= 1u << type;
            }
        }
        if (world <= 1) {
            if (rid < U) {
#pragma unroll
                for (int type = 0; type < 4; ++type) {
                    A[4 * rid + type] = hs[type]; V[4 * rid + type] = (u32)(4 * rid + type);
                    if (B) B[4 * rid + type] = ks[type];
                }
            }
            continue;
        }
        const u32 cnt = (u32)__popc(own);
        u32 inc = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const u32 y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        if (threadIdx.x == 0) {
            u32 tot = 0;
            for (int w = 0; w < 8; ++w) { const u32 x = s_warp[w]; s_warp[w] = tot; tot += x; }
            s_base = tot ? atomicAdd(n_out, (unsigned long long)tot) : 0ull;
        }
        __syncthreads();
        u64 pos = s_base + s_warp[warp] + (inc - cnt);
        if (pos + cnt <= room) {        // else: the host sees n_out > room and repeats the pass with room for all
#pragma unroll
            for (int type = 0; type < 4; ++type)
                if (own & (1u << type)) { A[pos] = hs[type]; V[pos] = (u32)(4 * rid + type); if (B) B[pos] = ks[type]; ++pos; }
        }
        __syncthreads();
    }
}

// pass 1 over the bucketed records, first round: claim the first empty slot of the key's home sector when no slot before it
// carries the key's tag -- the case of every key that is new to the index (a key lives in the first slot that was empty
// when it arrived, and slots are never freed: having reached an empty slot, the key is not in the index).  A short chain of
// dependent accesses (record, sector, CAS) and no divergence; everything else (tag seen, sector full, CAS lost) is appended
// to the block's segment of `retry` for the second round.
// While the records are inserted, a slot's payload is the index of its representative's RECORD: a tag match is confirmed
// from that record (same bucket, L2-resident while the bucket is worked on) instead of the reads.  table_runs_kernel puts
// the entries in place afterwards.
__global__ void __launch_bounds__(256) table_claim_kernel(const u64 *__restrict__ A, u64 n_rec,
                                                           u64 *__restrict__ slots, u64 nsec, u32 *__restrict__ where,
                                                           u32 *__restrict__ retry, u32 *__restrict__ n_retry)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    bool again = false;
    if (i < n_rec) {
        const u64 hsh = A[i];
        const u64 tag = slot_tag(hsh);
        const u64 sec = home_sector(hsh, nsec);
        u64 *sp = slots + kSlotsPerSector * sec;
        const ulonglong2 lo = __ldcg(reinterpret_cast<const ulonglong2 *>(sp)), hi = __ldcg(reinterpret_cast<const ulonglong2 *>(sp) + 1);
        const u64 cur[4] = { lo.x, lo.y, hi.x, hi.y };
        int q = -1;
        bool seen = false;
#pragma unroll
        for (int x = 3; x >= 0; --x) {
            if (cur[x] == 0) { q = x; seen = false; }                      // tags before the FIRST empty slot are what counts
            else if (slot_get_tag(cur[x]) == tag) seen = true;
        }
        again = true;
        if (q >= 0 && !seen) {
            const u64 old = atomicCAS((unsigned long long *)(sp + q), 0ull, (unsigned long long)slot_encode(hsh, 1, i));
            if (old == 0) { where[i] = (u32)(kSlotsPerSector * sec + q); again = false; }
        }
    }
    // the block's failures, compacted behind each other in its own 256-entry segment of `retry` (a global cursor would be
    // one atomic per warp on a single address: 3.5 M of them serialise to 9 ms at cfg4)
    __shared__ u32 s_cnt[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned m = __ballot_sync(0xffffffffu, again);
    if (lane == 0) s_cnt[warp] = (u32)__popc(m);
    __syncthreads();
    u32 base = 0, total = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) { if (w < warp) base += s_cnt[w]; total += s_cnt[w]; }
    if (again) retry[(u64)blockIdx.x * 256 + base + __popc(m & ((1u << lane) - 1u))] = (u32)i;
    if (threadIdx.x == 0) n_retry[blockIdx.x] = total;
}

// second round: the whole find-or-claim loop of table_insert_kernel on the records of `retry`; a tag match is confirmed by the
// hash and v0 of the representative's record (see table_keys_kernel)
__global__ void __launch_bounds__(64) table_insert_sorted_kernel(const u64 *__restrict__ A, const u64 *__restrict__ B, const u32 *__restrict__ retry,
                                                                   const u32 *__restrict__ n_retry,
                                                                   u64 *__restrict__ slots, u64 nsec, u32 *__restrict__ where, u32 *__restrict__ overflow)
{
    // block b (64 threads: 32 such blocks fill an SM's warp slots) takes the failures of block b of the first round: dense
    // warps, no list to assemble
    const u32 mine = n_retry[blockIdx.x];
    for (u32 k = threadIdx.x; k < mine; k += blockDim.x) {
        const u64 i = retry[(u64)blockIdx.x * 256 + k];
        const u64 hsh = A[i];
        const u64 v0 = B ? B[i] : 0ull;
        const u64 tag = slot_tag(hsh);
        u64 sec = home_sector(hsh, nsec);
        bool done = false;
        u64 tries = 0;
        while (!done) {
            for (int q = 0; q < kSlotsPerSector && !done; ++q) {
                u64 *sp = slots + kSlotsPerSector * sec + q;
                u64 cur = load_slot(sp);
                if (cur == 0) {
                    const u64 old = atomicCAS((unsigned long long *)sp, 0ull, (unsigned long long)slot_encode(hsh, 1, i));
                    if (old == 0) { where[i] = (u32)(kSlotsPerSector * sec + q); done = true; break; }
                    cur = old;
                }
                if (slot_get_tag(cur) != tag) continue;
                const u64 rep = slot_get_payload(cur);
                if (A[rep] != hsh || (B && B[rep] != v0)) continue;
                while (slot_get_count(cur) < 127) {
                    const u64 old = atomicCAS((unsigned long long *)sp, (unsigned long long)cur, (unsigned long long)(cur + kCountOne));
                    if (old == cur) break;
                    cur = old;
                }
                where[i] = (u32)(kSlotsPerSector * sec + q);
                done = true;
            }
            sec = (sec + 1 == nsec) ? 0 : sec + 1;
            if (++tries > nsec) { *overflow = 1; where[i] = kNotOwned; break; }
        }
    }
}

// pass 3 over the bucketed records
__global__ void __launch_bounds__(256) table_fill_sorted_kernel(const u64 *__restrict__ slots, const u32 *__restrict__ where, const u32 *__restrict__ V, u64 n_rec,
                                                                 u32 *__restrict__ cursor, u32 *__restrict__ entries)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_rec; i += (u64)gridDim.x * blockDim.x) {
        if (where[i] == kNotOwned) continue;
        const u64 v = slots[where[i]];
        const u32 c = slot_get_count(v);
        if (c < 2 || c >= (u32)kHashThreshold) continue;
        const u64 off = slot_get_payload(v);
        entries[off + atomicAdd(&cursor[off], 1u)] = V[i];
    }
}

// pass 2a: run length of every slot that owns a run in entries[]; distinct / masked key counters.  Bucketed build (recV):
// the payload of a slot without a run, a record index so far, becomes the representative's entry (the record's slot
// neighbours have neighbouring hashes, so recV is read within one bucket's range)
__global__ void __launch_bounds__(256) table_runs_kernel(u64 *__restrict__ slots, u64 cap, const u32 *__restrict__ recV, u32 *__restrict__ run,
                                                          unsigned long long *counters)
{
    unsigned long long distinct = 0, over = 0;
    for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += (u64)gridDim.x * blockDim.x) {
        const u64 v = slots[s];
        const u32 c = v ? slot_get_count(v) : 0u;
        const bool has_run = c >= 2 && c < (u32)kHashThreshold;
        run[s] = has_run ? c : 0u;
        if (recV && v && !has_run) slots[s] = (v & ~0x1FFFFFFFFull) | (u64)recV[slot_get_payload(v)];
        distinct += v != 0;
        over += c >= (u32)kHashThreshold;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { distinct += __shfl_xor_sync(0xffffffffu, distinct, o); over += __shfl_xor_sync(0xffffffffu, over, o); }
    if ((threadIdx.x & 31) == 0) { if (distinct) atomicAdd(&counters[0], distinct); if (over) atomicAdd(&counters[1], over); }
}

// pass 2b: payload of run-owning slots := offset of the run
__global__ void __launch_bounds__(256) table_offsets_kernel(u64 *__restrict__ slots, u64 cap, const u32 *__restrict__ run, const u32 *__restrict__ off)
{
    for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += (u64)gridDim.x * blockDim.x)
        if (run[s]) slots[s] = (slots[s] & ~0x1FFFFFFFFull) | (u64)off[s];
}

// pass 3: entries of run-owning keys take the next free position of their run
__global__ void __launch_bounds__(256) table_fill_kernel(const u64 *__restrict__ slots, const u32 *__restrict__ where, u64 n,
                                                          u32 *__restrict__ cursor, u32 *__restrict__ entries)
{
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (u64)gridDim.x * blockDim.x) {
        if (where[t] == kNotOwned) continue;
        const u64 v = slots[where[t]];
        const u32 c = slot_get_count(v);
        if (c < 2 || c >= (u32)kHashThreshold) continue;
        const u64 off = slot_get_payload(v);
        entries[off + atomicAdd(&cursor[off], 1u)] = (u32)t;
    }
}

// pass 4: bucket order = (readId asc, type asc) = entry value ascending
__global__ void __launch_bounds__(256) table_order_kernel(const u64 *__restrict__ slots, u64 cap, u32 *__restrict__ entries)
{
    for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += (u64)gridDim.x * blockDim.x) {
        const u64 v = slots[s];
        if (v == 0) continue;
        const u32 c = slot_get_count(v);
        if (c < 2 || c >= (u32)kHashThreshold) continue;
        u32 *e = entries + slot_get_payload(v);
        for (u32 a = 1; a < c; ++a) {
            const u32 x = e[a];
            u32 b = a;
            while (b > 0 && e[b - 1] > x) { e[b] = e[b - 1]; --b; }
            e[b] = x;
        }
    }
}

static unsigned big_grid(u64 n, unsigned block = 256)
{
    unsigned g = grid_for(n, block, 4);
    return g > kSMs * 16u ? kSMs * 16u : g;
}

u64 table_shard_slots(u64 U, int world)
{
    // load factor <= 2/3 even if all 4U keys are distinct (typically ~0.5)
    // (a shard expects 1/world of the keys; 10 % head room for the imbalance of the split)
    const u64 n = 4 * U;
    u64 nsec = (n + n / 2 + kSlotsPerSector - 1) / kSlotsPerSector;
    if (world > 1) nsec = nsec / (u64)world + nsec / (10 * (u64)world) + 1;
    if (nsec < 256) nsec = 256;
    return nsec * kSlotsPerSector;
}

// rank / world: the key-hash shard this context holds (0 / 1 = the whole table).  A shard indexes only the keys
// with key_owner(hash) == rank; every context still streams all 4U entries (the reads are replicated).
void stage_build_table(Context &c, int rank, int world, bool joint)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    SG_CHECK(c.have_reads, "organize_reads must run before build_hash_table");
    SG_CHECK(world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world, "bad rank / world");
    c.tb_rank = rank; c.tb_world = world; c.tb_shards = 1; c.tb_entries = 0; c.tb_joint = joint && world > 1;
    const u64 U = c.cnt.unique_reads;
    const int SW = c.SW, h = c.h;
    c.cnt.distinct_keys = 0; c.cnt.keys_over_threshold = 0; c.cap = 0; c.cnt.table_capacity = 0;
    if (U == 0) { c.slots.release(); c.entries.release(); c.have_table = true; return; }
    const u64 n = 4 * U;
    SG_CHECK(n < 0xFFFFFFFFull, "at most 2^30-1 unique reads per context");
    const u64 cap = table_shard_slots(U, world), nsec = cap / kSlotsPerSector;
    SG_CHECK(cap < 0xFFFFFFFFull, "slot index too large for one context");
    // joint: the shard is built in its place inside an array with room for all shards (stage_table_gather_* completes it)
    c.slots.alloc(c.tb_joint ? cap * (u64)world : cap, st);
    u64 *const slots = c.slots.p + (c.tb_joint ? (u64)rank * cap : 0);
    DevBuf<u32> &entries = c.tb_joint ? c.entries_loc : c.entries;
    SG_CUDA(cudaMemsetAsync(slots, 0, cap * sizeof(u64), st));

    // bucketed build when the index is far larger than L2 (see the header); SAGE2GPU_TABLE_BUILD=direct|bucketed overrides
    const char *env = getenv("SAGE2GPU_TABLE_BUILD");
    const int forced = !env ? 0 : (env[0] == 'd' ? 1 : 2);
    // (not in low-memory mode: the records take 2.75 x (h > 32: 3.75 x) the workspace of the direct build, and config #5 fits
    // 180 GB with nothing to spare)
    const bool bucketed = forced ? forced == 2 : (!c.opt_low_memory && cap * sizeof(u64) >= ((size_t)256 << 20));
    DevBuf<u32> where, d_overflow(1, st), v0, v1;
    DevBuf<u64> a0, a1, b0, b1;
    const bool with_v0 = h > 32;       // v0 is always 0 otherwise (table_keys_kernel)
    const u32 *recV = nullptr;
    u64 n_rec = n;
    SG_CUDA(cudaMemsetAsync(d_overflow.p, 0, sizeof(u32), st));
    if (!bucketed) {
        where.alloc(n, st);
        table_insert_kernel<<<big_grid(n), 256, 0, st>>>(c.F.p, c.RC.p, c.len.p, U, SW, c.SWS, h, slots, nsec, where.p, rank, world, d_overflow.p);
        SG_LAUNCHED();
    } else {
        u64 room = world > 1 ? n / (u64)world + n / (4 * (u64)world) + 4096 : n;      // owned records: 1/world of all, 25 % head room
        if (const char *e = getenv("SAGE2GPU_TABLE_ROOM")) { if (world > 1) room = (u64)atoll(e); }      // test knob: force the second round
        DevBuf<unsigned long long> d_nrec(1, st);
        for (;;) {
            a0.alloc(room + 1, st); v0.alloc(room + 1, st);
            if (with_v0) b0.alloc(room + 1, st);
            SG_CUDA(cudaMemsetAsync(d_nrec.p, 0, sizeof(unsigned long long), st));
            table_keys_kernel<<<big_grid(U), 256, 0, st>>>(c.F.p, c.RC.p, c.len.p, U, SW, c.SWS, h, rank, world, a0.p, b0.p, v0.p, room, d_nrec.p);
            SG_LAUNCHED();
            if (world <= 1) break;
            unsigned long long h_nrec = 0;
            SG_CUDA(cudaMemcpyAsync(&h_nrec, d_nrec.p, sizeof(h_nrec), cudaMemcpyDeviceToHost, st));
            SG_CUDA(cudaStreamSynchronize(st));
            n_rec = h_nrec;
            if (n_rec <= room) break;
            room = n_rec;               // a very uneven key split (one key in most reads): once more with room for all of them
        }
        a1.alloc(n_rec + 1, st); v1.alloc(n_rec + 1, st);
        if (with_v0) b1.alloc(n_rec + 1, st);
        SortCols cols;
        cols.a[0] = a0.p; cols.a[1] = a1.p; cols.b[0] = b0.p; cols.b[1] = b1.p; cols.v[0] = v0.p; cols.v[1] = v1.p;
        const int cur = radix_sort_bits(cols, 0, n_rec, false, 56, 64, st);
        recV = cols.v[cur];
        where.alloc(n_rec + 1, st);
        // one record per thread: the blocks start in record order, so the records in flight span about one bucket (a capped grid
        // with a grid-stride loop drifts apart over its ~200 rounds and loses the locality)
        if (n_rec) {
            const unsigned blocks = grid_for(n_rec, 256);
            DevBuf<u32> retry((u64)blocks * 256, st), n_retry(blocks, st);
            table_claim_kernel<<<blocks, 256, 0, st>>>(cols.a[cur], n_rec, slots, nsec, where.p, retry.p, n_retry.p);
            SG_LAUNCHED();
            table_insert_sorted_kernel<<<blocks, 64, 0, st>>>(cols.a[cur], cols.b[cur], retry.p, n_retry.p, slots, nsec, where.p, d_overflow.p);
            SG_LAUNCHED();
            if (stage_stats_enabled()) {
                std::vector<u32> h_retry(blocks);
                SG_CUDA(cudaMemcpyAsync(h_retry.data(), n_retry.p, blocks * sizeof(u32), cudaMemcpyDeviceToHost, st));
                SG_CUDA(cudaStreamSynchronize(st));
                u64 tot = 0;
                for (u32 x : h_retry) tot += x;
                fprintf(stderr, "sage2gpu stats: build_table records=%llu retry_records=%llu\n", (unsigned long long)n_rec, (unsigned long long)tot);
            }
        }
    }

    DevBuf<u32> run(cap, st), off(cap, st), d_total(1, st);
    DevBuf<unsigned long long> d_cnt(2, st);
    SG_CUDA(cudaMemsetAsync(d_cnt.p, 0, 2 * sizeof(unsigned long long), st));
    table_runs_kernel<<<big_grid(cap), 256, 0, st>>>(slots, cap, recV, run.p, d_cnt.p);
    SG_LAUNCHED();
    exclusive_scan_u32(run.p, off.p, cap, d_total.p, st);
    u32 M = 0;
    unsigned long long h_cnt[2];
    u32 h_overflow = 0;
    SG_CUDA(cudaMemcpyAsync(&h_overflow, d_overflow.p, sizeof(u32), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaMemcpyAsync(&M, d_total.p, sizeof(u32), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaMemcpyAsync(h_cnt, d_cnt.p, sizeof(h_cnt), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    SG_CHECK(h_overflow == 0, "slot index of this table shard is full (key split too uneven)");

    entries.alloc(M, st);
    c.tb_entries = M;
    if (M) {
        table_offsets_kernel<<<big_grid(cap), 256, 0, st>>>(slots, cap, run.p, off.p);
        SG_LAUNCHED();
        DevBuf<u32> cursor(M, st);
        SG_CUDA(cudaMemsetAsync(cursor.p, 0, (size_t)M * sizeof(u32), st));
        if (bucketed) table_fill_sorted_kernel<<<grid_for(n_rec, 256), 256, 0, st>>>(slots, where.p, recV, n_rec, cursor.p, entries.p);
        else table_fill_kernel<<<big_grid(n), 256, 0, st>>>(slots, where.p, n, cursor.p, entries.p);
        SG_LAUNCHED();
        table_order_kernel<<<big_grid(cap), 256, 0, st>>>(slots, cap, entries.p);
        SG_LAUNCHED();
        SG_CUDA(cudaStreamSynchronize(st));     // cursor / where lifetimes end here
    }
    c.cap = cap;
    c.cnt.table_capacity = cap;
    c.cnt.distinct_keys = h_cnt[0];
    c.cnt.keys_over_threshold = h_cnt[1];
    c.have_table = true;
}

// ---- several GPUs, replicated table: every rank builds one key-hash shard, the shards are all-gathered ---------------
// layout: room for all shards back to back (equal slot counts; entry runs of shard q behind those of shards < q), this
// rank's shard moved to its place; the host all-gathers both arrays; finish: the run offsets stored in the slots of
// shard q become offsets into the joint entries[] array.
__global__ void __launch_bounds__(256) table_rebase_kernel(u64 *__restrict__ slots, u64 cap_shard, u64 ebase)
{
    for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < cap_shard; s += (u64)gridDim.x * blockDim.x) {
        const u64 v = slots[s];
        if (v == 0) continue;
        const u32 c = slot_get_count(v);
        if (c >= 2 && c < (u32)kHashThreshold) slots[s] = (v & ~0x1FFFFFFFFull) | (slot_get_payload(v) + ebase);
    }
}

void stage_table_gather_layout(Context &c, const u64 *entry_counts, void **slots, void **entries, u64 *slots_per_shard, u64 *entries_first)
{
    cudaStream_t st = c.stream;
    SG_CHECK(c.have_table && c.tb_world > 1 && c.tb_shards == 1, "sage2gpu_build_hash_table_shard must run first");
    SG_CHECK(entry_counts && entry_counts[c.tb_rank] == c.tb_entries, "this rank's entry count does not match its shard");
    const int world = c.tb_world;
    const u64 cap_shard = c.cap;
    u64 tot = 0, base = 0;
    for (int q = 0; q < world; ++q) { if (q < c.tb_rank) base += entry_counts[q]; tot += entry_counts[q]; }
    SG_CHECK(tot < 0xFFFFFFFFull && cap_shard * (u64)world < (1ull << 40), "table too large");
    SG_CHECK(c.tb_joint, "the shard must be built with sage2gpu_build_hash_table_part for the gather");
    c.entries.alloc(tot, st);
    if (c.tb_entries) SG_CUDA(cudaMemcpyAsync(c.entries.p + base, c.entries_loc.p, (size_t)c.tb_entries * sizeof(u32), cudaMemcpyDeviceToDevice, st));
    SG_CUDA(cudaStreamSynchronize(st));
    if (slots) *slots = c.slots.p;
    if (entries) *entries = c.entries.p;
    if (slots_per_shard) *slots_per_shard = cap_shard;
    if (entries_first) *entries_first = base;
}

void stage_table_gather_finish(Context &c, const u64 *entry_counts, const u64 *distinct, const u64 *over)
{
    cudaStream_t st = c.stream;
    SG_CHECK(c.have_table && c.tb_world > 1 && c.tb_shards == 1 && entry_counts, "sage2gpu_table_gather_layout must run first");
    const int world = c.tb_world;
    const u64 cap_shard = c.cap;
    u64 ebase = 0, d = 0, o = 0;
    for (int q = 0; q < world; ++q) {
        if (ebase) { table_rebase_kernel<<<big_grid(cap_shard), 256, 0, st>>>(c.slots.p + (size_t)q * cap_shard, cap_shard, ebase); SG_LAUNCHED(); }
        ebase += entry_counts[q];
        if (distinct) d += distinct[q];
        if (over) o += over[q];
    }
    c.tb_entries = ebase;
    c.tb_shards = world; c.tb_world = 1; c.tb_rank = 0;
    c.cap = cap_shard * (u64)world;
    c.cnt.table_capacity = c.cap;
    if (distinct) c.cnt.distinct_keys = d;
    if (over) c.cnt.keys_over_threshold = o;
}

}  // namespace sg
