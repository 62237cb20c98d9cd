// search_common.cuh -- pieces shared by the phase-A / phase-C search kernels (search.cu) and the superstring fast path of
// phase A (search_fast.cu): launch parameters, 256-bit loads, key extraction, the funnel-shift window and the
// sector-index probe (HashTable::hashTableSearch, hashTable.cpp:193-231).
#pragma once
#include "context.h"

namespace sg {

struct SearchParams {
    const u64 *F, *RC;
    const u64 *slots;
    const u32 *entries;
    u64 nsec, U;        // nsec: sectors of one shard of the slot index (of the whole index when shards == 1)
    int shards;         // key-hash shards the index is assembled from (stage_table_gather_*)
    u64 lo, hi;         // phase A handles read indices [lo, hi)
    int h, k;
    // ROUTED kernels (sharded table, shard.cu): the probes of a batch of reads were answered by the shards that
    // own their keys.  The batch is ids[0..n) (0-based read indices) or lo + [0..n); the answer word of window j
    // of the s-th read is wslot[s * wstride + j] (core.cuh answer_encode) and `entries` is the batch's own entry
    // stream.  Untrusted answers (tag probes) are proven in the kernel; a collision sets redo[s] and skips the read.
    const u64 *wslot;
    const u32 *ids;
    uint8_t *redo;
    u64 n;
    u32 wstride;
    int trusted;
    // phase_a_kernel (not ROUTED): number of ids when it is only known on the device (the redo list of search_fast.cu);
    // nullptr: ids[0..hi-lo), or [lo, hi) in id order when ids is nullptr too
    const unsigned *n_dev;
};

// 256-bit read-only load: one 32-byte sector per lane and instruction (LDG.E.256 on sm_100a)
__device__ __forceinline__ void ldg256(const u64 *p, u64 (&v)[4])
{
    asm volatile("ld.global.nc.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v[0]), "=l"(v[1]), "=l"(v[2]), "=l"(v[3]) : "l"(p));
}
// the same with an L2 eviction priority: the slot index is re-read by every read (keep: evict_last), a partner record
// is needed once per overlap and should not push the index out (evict_first)
__device__ __forceinline__ void ldg256_keep(const u64 *p, u64 (&v)[4])
{
    asm volatile("ld.global.nc.L2::evict_last.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v[0]), "=l"(v[1]), "=l"(v[2]), "=l"(v[3]) : "l"(p));
}
__device__ __forceinline__ void ldg256_stream(const u64 *p, u64 (&v)[4])
{
    asm volatile("ld.global.nc.L2::evict_first.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v[0]), "=l"(v[1]), "=l"(v[2]), "=l"(v[3]) : "l"(p));
}

template <int SW>
struct SearchCfg {
    static constexpr int WARPS = SW <= 8 ? 8 : (SW <= 16 ? 4 : 2);
    static constexpr int SWS = SW <= 4 ? 4 : (SW <= 8 ? 8 : (SW <= 16 ? 16 : 32));   // == storage_words(SW): F / RC stride
    static constexpr int LPI = SWS / 4;          // lanes that fetch one partner record together (one sector each)
    static constexpr int SWP = SWS + 1;          // odd record stride in shared memory (bank spread) + the word read past
};

// Grid of a warp-per-read kernel with a grid-stride loop: one warp per read, at most blocks_per_sm blocks per SM, at least
// one block.
inline unsigned search_grid(u64 n_reads, int warps, int blocks_per_sm)
{
    u64 g = (n_reads + warps - 1) / warps;
    const u64 cap = (u64)kSMs * blocks_per_sm;
    if (g > cap) g = cap;
    if (g == 0) g = 1;
    return (unsigned)g;
}

// search_grid for a persistent launch of KERNEL: as many blocks per SM as can be resident at once (occupancy API, asked
// once per kernel).
template <auto KERNEL>
unsigned persistent_grid(u64 n_reads, int warps)
{
    static int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        SG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, KERNEL, warps * 32, 0));
        if (blocks_per_sm < 1) blocks_per_sm = 1;
    }
    return search_grid(n_reads, warps, blocks_per_sm);
}

template <int SW>
__device__ __forceinline__ u64 t_window32(const u64 *X, int s)
{
    const int i = s >> 5, sh = (s & 31) * 2;
    const u64 a = i < SW ? X[i] : 0ull;
    const u64 b = (i + 1) < SW ? X[i + 1] : 0ull;
    return sh == 0 ? a : ((a << sh) | (b >> (64 - sh)));
}

template <int SW>
__device__ __forceinline__ void t_extract_key(const u64 *X, int j, int h, u64 &v0, u64 &v1)
{
    if (h <= 32) { v0 = 0; v1 = t_window32<SW>(X, j) >> (64 - 2 * h); }
    else { v0 = t_window32<SW>(X, j) >> (64 - 2 * (h - 32)); v1 = t_window32<SW>(X, j + h - 32); }
}

// masks of the first h bases (the hash key) inside the first two words of a compare
__device__ __forceinline__ void key_masks(int h, u64 &km0, u64 &km1)
{
    km0 = h >= 32 ? ~0ull : ~(~0ull >> (2 * h));
    km1 = h <= 32 ? 0ull : (h >= 64 ? ~0ull : ~(~0ull >> (2 * (h - 32))));
}

// 64 bits starting `s` bits (0..63) into the 128-bit string a:b, by two 32-bit funnel shifts
__device__ __forceinline__ u64 funnel64(u64 a, u64 b, bool upper, unsigned s5)
{
    const u32 ah = (u32)(a >> 32), al = (u32)a, bh = (u32)(b >> 32), bl = (u32)b;
    const u32 x0 = upper ? al : ah, x1 = upper ? bh : al, x2 = upper ? bl : bh;
    return ((u64)__funnelshift_l(x1, x0, s5) << 32) | __funnelshift_l(x2, x1, s5);
}

// hashTableSearch (hashTable.cpp:193-231) on the sector index.  cnt == 0: absent (or masked).
// `exact`: confirm every tag match by re-extracting the key from the bucket's first read (:203-220);
// otherwise only masked keys are confirmed here and the caller proves the key in stage 2.
template <int SW>
__device__ __forceinline__ void probe_window(const SearchParams &P, u64 v0, u64 v1, bool exact, u64 &payload, u32 &cnt)
{
    payload = 0; cnt = 0;
    const u64 hsh = hash_key(v0, v1);
    const u64 tag = slot_tag(hsh);
    const u64 sbase = shard_base_sector(hsh, P.nsec, P.shards);
    u64 sec = home_sector(hsh, P.nsec);
    for (;;) {
        u64 s[4];
        ldg256_keep(P.slots + kSlotsPerSector * (sbase + sec), s);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const u64 slot = s[t];
            if (slot == 0) return;
            if (slot_get_tag(slot) != tag) continue;
            const u32 c = slot_get_count(slot);
            if (exact || c >= (u32)kHashThreshold) {
                const u32 ent = (c == 1 || c >= (u32)kHashThreshold) ? (u32)slot_get_payload(slot) : __ldg(&P.entries[slot_get_payload(slot)]);
                const u64 rid = ent >> 2;
                const int type = (int)(ent & 3);
                const u64 *X = ((type & 2) ? P.RC : P.F) + rid * SearchCfg<SW>::SWS;
                const int l = (int)(__ldg(&X[SW - 1]) & 0xFFFF);
                u64 w0, w1;
                t_extract_key<SW>(X, (type & 1) ? l - P.h : 0, P.h, w0, w1);
                if (w0 != v0 || w1 != v1) continue;            // tag collision: keep probing
                if (c >= (u32)kHashThreshold) return;         // masked key reads as absent (:203)
            }
            payload = slot_get_payload(slot); cnt = c;
            return;
        }
        sec = (sec + 1 == P.nsec) ? 0 : sec + 1;
    }
}

}  // namespace sg
