// search_fast.cu -- K4, phase A of EconomyGraph::buildInitialOverlapGraph (economyGraph/economyGraph.cpp:64-452), for
// the reads whose hits all agree: the SUPERSTRING scan.  search.cu's phase_a_kernel stays the general path (hit-by-hit
// chain, restarts after tag collisions, any number of windows and bucket entries) and runs afterwards on the reads this
// kernel could not certify (a list built on the device; 0 of 2.24 M reads at cfg2, 4,008 of 27.9 M at cfg4).
//
// One warp per read.
//   1. PROBE    all windows of the read first: lane l derives the key of window base+l by funnel shifts, reads ONE
//               32-byte sector of the slot index and picks its slot without branches; the (window, bucket entry) items
//               are written to shared memory in the reference's order (window ascending, bucket order).
//   2. COMPARE  32 items per round, one partner record per lane (fetched by lane groups, one 256-bit load per sector).
//               Per side the warp keeps a superstring S in shared memory: read i (right hits) or its reverse complement
//               (left hits) followed by the bases the hits seen so far agree on beyond its end.  An item is compared
//               ONCE, against S: the position of the first difference tells everything --
//                   inside the key            -> 24-bit tag collision (first entry of a bucket): the general path redoes the read
//                   inside read i's span      -> not an overlap (compareStringInBytes == 0, economyGraph.cpp:712-758)
//                   beyond read i's end       -> a hit that contradicts an earlier hit: not certifiable here
//                   none                      -> a hit, consistent with every hit before it
//   3. EXTEND   of the hits of a round the one reaching furthest appends its new bases to S (a few lanes, one word
//               each) and the other hits of that side are checked on the part S did not cover before.
// If no hit contradicts S and no window holds two hits of one side, every adjacent pair of hits is consistent, so the
// reference's chain (economyGraph.cpp:94-437) never sets itsAmbig and never takes its second-hit-in-a-window branches:
// rightExtension = the first right hit, leftExtension = the last left hit, connections = the number of hits.
// tests/host_emul.cpp restates this scan on the CPU (fast_certify) and checks it against the oracle.
#include <stdlib.h>
#include "search_common.cuh"

namespace sg {

constexpr int kFastCap = 192;        // items (window, bucket entry) of one read held in shared memory
constexpr int kFastWindows = 128;    // windows of one read (the window travels in 7 bits)

// hashTableSearch (hashTable.cpp:193-231) on the sector index with a branch-free sector test: the slots of a sector fill
// in order, so empty slots are a suffix and "no tag match + an empty slot" means absent.  A tag match counts as found
// (proven by the compare of the bucket's first entry).  Returns false for a masked key (>= 100 entries), which
// probe_window confirms through its representative read.
__device__ __forceinline__ bool probe_sectors(const SearchParams &P, u64 hsh, u64 &payload, u32 &cnt)
{
    const u64 tag = slot_tag(hsh);
    const u64 *shard = P.slots + kSlotsPerSector * shard_base_sector(hsh, P.nsec, P.shards);
    u64 sec = home_sector(hsh, P.nsec);
    payload = 0; cnt = 0;
    for (;;) {
        u64 s[4];
        ldg256_keep(shard + kSlotsPerSector * sec, s);
        const bool m0 = (s[0] >> 40) == tag && s[0] != 0, m1 = (s[1] >> 40) == tag && s[1] != 0;
        const bool m2 = (s[2] >> 40) == tag && s[2] != 0, m3 = (s[3] >> 40) == tag && s[3] != 0;
        const u64 cand = m0 ? s[0] : (m1 ? s[1] : (m2 ? s[2] : (m3 ? s[3] : 0ull)));
        if (cand != 0) {
            const u32 c = slot_get_count(cand);
            if (c >= (u32)kHashThreshold) return false;
            payload = slot_get_payload(cand); cnt = c;
            return true;
        }
        if (s[3] == 0) return true;                  // room left in this sector: the key is absent
        sec = (sec + 1 == P.nsec) ? 0 : sec + 1;
    }
}

// Position of the first base t in [0, ov) with S[s + t] != Y[t]; 0x7fffffff when there is none.
template <int SW>
__device__ __forceinline__ int first_mismatch(const u64 *S, int s, const u64 *Y, int ov)
{
    const int wb = ov >> 5;
    const u64 bm = ~(~0ull >> ((ov & 31) * 2));          // 0 when ov is a multiple of 32
    const int i0 = s >> 5;
    const unsigned sh = (unsigned)(s & 31) * 2;
    const bool upper = sh >= 32;
    const unsigned s5 = sh & 31;
    int fw = SW;
    u64 fd = 0;
    u64 a = S[i0];
#pragma unroll
    for (int w = 0; w < SW; ++w) {
        if (w <= wb) {
            const u64 b = S[i0 + w + 1];
            u64 d = funnel64(a, b, upper, s5) ^ Y[w];
            if (w == wb) d &= bm;
            if (d != 0 && fw == SW) { fw = w; fd = d; }
            a = b;
        }
    }
    return fw == SW ? 0x7fffffff : 32 * fw + (__clzll((long long)fd) >> 1);
}

// S[s + t] == Y[t] for t in [from, len2)  (from < len2)
__device__ __forceinline__ bool tail_equal(const u64 *S, int s, const u64 *Y, int from, int len2)
{
    const int w0 = from >> 5, wl = (len2 - 1) >> 5;
    const unsigned sh = (unsigned)(s & 31) * 2;
    const bool upper = sh >= 32;
    const unsigned s5 = sh & 31;
    const u64 *Sp = S + (s >> 5) + w0;
    u64 acc = 0;
    u64 a = Sp[0];
    for (int w = w0; w <= wl; ++w) {
        const u64 b = *++Sp;
        u64 d = funnel64(a, b, upper, s5) ^ Y[w];
        if (w == w0) d &= ~0ull >> ((from & 31) * 2);
        if (w == wl && (len2 & 31)) d &= ~(~0ull >> ((len2 & 31) * 2));
        acc |= d;
        a = b;
    }
    return acc == 0;
}

// 32 bases of a shared-memory row starting at base s >= 0, without bounds checks: the row holds word (s >> 5) + 1
// (superstring rows: two records and a word; partner rows: the storage stride and a word).  Bases past the data are
// garbage that callers mask off.
__device__ __forceinline__ u64 row_window32(const u64 *X, int s)
{
    const unsigned sh = (unsigned)(s & 31) * 2;
    return funnel64(X[s >> 5], X[(s >> 5) + 1], sh >= 32, sh & 31);
}

// t_extract_key on a row (the key lies inside the read, so the word after it is within the row)
__device__ __forceinline__ void row_extract_key(const u64 *X, int j, int h, u64 &v0, u64 &v1)
{
    if (h <= 32) { v0 = 0; v1 = row_window32(X, j) >> (64 - 2 * h); }
    else { v0 = row_window32(X, j) >> (64 - 2 * (h - 32)); v1 = row_window32(X, j + h - 32); }
}

// 32 bases of record M starting at base s (may be negative: bases before the record read as 0)
__device__ __forceinline__ u64 window_signed(const u64 *M, int s)
{
    if (s >= 0) return row_window32(M, s);
    if (s <= -32) return 0ull;
    return M[0] >> (2 * (-s));
}

template <int SW, int MINB>
__global__ void __launch_bounds__(SearchCfg<SW>::WARPS * 32, MINB)
phase_a_fast_kernel(SearchParams P, u64 *__restrict__ extR, u64 *__restrict__ extL, uint8_t *__restrict__ flag5,
                    u32 *__restrict__ cont_max, unsigned long long *__restrict__ counters, u32 *__restrict__ redo_ids,
                    unsigned *__restrict__ redo_count)
{
    constexpr int WARPS = SearchCfg<SW>::WARPS, SWP = SearchCfg<SW>::SWP, SWS = SearchCfg<SW>::SWS, LPI = SearchCfg<SW>::LPI, IPI = 32 / LPI;
    constexpr int SS = 2 * SW + 2;                  // words of one superstring: two records + the word read past
    constexpr unsigned FULL = 0xffffffffu;
    static_assert(SS <= 32, "the superstring is written one word per lane");
    __shared__ u64 sS[WARPS][2][SS];
    __shared__ u64 sQ[WARPS][32 * SWP];
    __shared__ u32 sEnt[WARPS][kFastCap];
    __shared__ uint8_t sWin[WARPS][kFastCap];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u64 *SR = sS[warp][0], *SL = sS[warp][1], *Qs = sQ[warp];
    u32 *ents = sEnt[warp];
    uint8_t *wins = sWin[warp];
    const u64 nwarps = (u64)gridDim.x * WARPS;
    const unsigned lt_mask = (1u << lane) - 1u;
    unsigned calls = 0, probes = 0;

    const u64 n_batch = P.hi - P.lo;
    for (u64 sb = (u64)blockIdx.x * WARPS + warp; sb < n_batch; sb += nwarps) {
        const u64 i = P.ids ? (u64)P.ids[sb] : P.lo + sb;
        // ---- the read and its reverse complement: the two superstrings' first len1 bases ----------------------
        u64 f = 0, r = 0;
        if (lane < SW) { f = P.F[i * SWS + lane]; r = P.RC[i * SWS + lane]; }
        const int len1 = (int)(__shfl_sync(FULL, f, SW - 1) & 0xFFFF);
        if (lane == SW - 1) { f &= ~0xFFFFull; r &= ~0xFFFFull; }       // the record keeps its length there
        __syncwarp();
        if (lane < SS) { SR[lane] = f; SL[lane] = r; }
        __syncwarp();
        const int W = len1 - P.h + 1;
        bool punt = W > kFastWindows;

        // ---- stage 1: probe every window, list the items ----------------------------------------------------
        // Two lists in one array: items of right entries (hash types 0 / 2) from the front, of left entries (1 / 3) from
        // the back.  The rounds take the right items from the LAST window down and then the left items from the FIRST
        // window up: the first hit of either side then reaches furthest, its bases complete the side's superstring in
        // one step, and the hits after it are single compares (fixed read length; anything else still works, slower).
        // Entries that need no compare (the read itself, a window outside the side's range, :94 / :279) are dropped here
        // unless they are the first of their bucket, which proves the bucket's key.
        int Tr = 0, Tl = 0;
        unsigned my_probes = 0;
        for (int base = 0; base < W && !punt; base += 32) {
            const int j = base + lane;
            u64 payload = 0;
            u32 cnt = 0;
            if (j < W) {
                u64 v0, v1;
                row_extract_key(SR, j, P.h, v0, v1);
                if (!probe_sectors(P, hash_key(v0, v1), payload, cnt)) probe_window<SW>(P, v0, v1, false, payload, cnt);
                my_probes++;
            }
            // The chunk's bucket sizes are scanned once; the warp then walks the chunk's entries 32 at a time, one per
            // lane (a bucket's entries are contiguous, so the loads are near-coalesced).  A lane finds its window by a
            // binary search over the scan, and the kept entries are compacted by ballot: both lists stay in window
            // order, then bucket order.
            u32 incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const u32 y = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += y; }
            const u32 excl = incl - cnt;
            const u32 tot = __shfl_sync(FULL, incl, 31);
            for (u32 t0 = 0; t0 < tot; t0 += 32) {
                const u32 t = t0 + lane;
                int lo = 0;
#pragma unroll
                for (int step = 16; step > 0; step >>= 1) {
                    const u32 pm = __shfl_sync(FULL, incl, lo + step - 1);
                    if (pm <= t) lo += step;
                }
                const u32 e = t - __shfl_sync(FULL, excl, lo), c = __shfl_sync(FULL, cnt, lo);
                const u64 pay = __shfl_sync(FULL, payload, lo);
                const int jw = base + lo;
                const bool valid = t < tot;
                u32 ent = 0;
                if (valid) ent = c == 1 ? (u32)pay : __ldg(&P.entries[pay + e]);
                const bool right = !(ent & 1u);
                const bool keep = valid && (e == 0 || ((ent >> 2) != (u32)i && (right ? gate_right(jw, len1, P.k) : gate_left(jw, P.k, P.h))));
                const unsigned kR = __ballot_sync(FULL, keep && right), kL = __ballot_sync(FULL, keep && !right);
                const int nR = __popc(kR), nL = __popc(kL);
                if (Tr + Tl + nR + nL > kFastCap) { punt = true; break; }
                if (keep) {
                    const int at = right ? Tr + __popc(kR & lt_mask) : kFastCap - 1 - (Tl + __popc(kL & lt_mask));
                    ents[at] = ent;
                    wins[at] = (uint8_t)(jw | (e == 0 ? 0x80 : 0));
                }
                Tr += nR; Tl += nL;
            }
        }
        const int T = Tr + Tl;
        __syncwarp();

        // ---- stages 2 + 3: rounds of 32 items ---------------------------------------------------------------
        int lenSR = len1, lenSL = len1, lastJR = -1, lastJL = -1;
        u32 connections = 0;
        unsigned my_calls = 0;
        int myRj = 0x7fffff, myLj = -1;                  // this lane's right hit with the smallest / left hit with the largest window
        u32 myRrid = 0, myRtl = 0, myLrid = 0, myLtl = 0;     // partner, type << 16 | length
        for (int r0 = 0; r0 < T && !punt; r0 += 32) {
            const int x = r0 + lane;
            const bool valid = x < T;
            const int idx = x < Tr ? Tr - 1 - x : kFastCap - 1 - (x - Tr);
            const u32 ent = valid ? ents[idx] : 0u;
            const int win = valid ? (int)wins[idx] : 0;
            const int jj = win & 127;
            const bool first = (win & 0x80) != 0;
            const u32 rid2 = ent >> 2;
            const int type = (int)(ent & 3);
            const bool right = !(type & 1);
            const bool need = valid && rid2 != (u32)i && (right ? gate_right(jj, len1, P.k) : gate_left(jj, P.k, P.h));
            const bool load = need || (valid && first);
            const u64 *rec = (partner_uses_rc(type) ? P.RC : P.F) + (u64)rid2 * SWS;
            // partner records -> shared memory, LPI lanes per record with one 256-bit load each
#pragma unroll
            for (int a = 0; a < LPI; ++a) {
                const int src = IPI * a + lane / LPI, part = lane % LPI;
                const u64 *base = reinterpret_cast<const u64 *>(__shfl_sync(FULL, (unsigned long long)rec, src));
                const bool fetch = __shfl_sync(FULL, (int)load, src) != 0 && 4 * part < SW;
                if (fetch) {
                    u64 v[4];
                    ldg256_stream(base + 4 * part, v);
#pragma unroll
                    for (int w = 0; w < 4; ++w) Qs[src * SWP + 4 * part + w] = v[w];
                }
            }
            __syncwarp();
            const u64 *Y = Qs + lane * SWP;
            bool hit = false, bad = false;
            int len2 = 0, s = 0, reach = 0;
            if (load) {
                len2 = (int)(Y[SW - 1] & 0xFFFF);
                s = right ? jj : len1 - jj - P.h;
                const int xlen = len1 - s;                         // bases of the partner inside read i's span
                const bool contained = len2 <= xlen;
                const int lenS = right ? lenSR : lenSL;
                const int ov = min(len2, lenS - s);
                const int tbad = first_mismatch<SW>(right ? SR : SL, s, Y, ov);
                if (first && tbad < P.h) bad = true;               // tag collision: the general path restarts with verified probes
                if (need) {
                    my_calls++;
                    const bool ok = tbad >= min(xlen, len2);
                    if (ok && contained) atomicMax(&cont_max[rid2], (u32)(i + 1));      // economyGraph.cpp:735
                    hit = ok && !contained;
                    if (hit && tbad < ov) bad = true;              // contradicts an earlier hit
                    reach = s + len2;
                }
            }
            // at most one hit per side and window
            const unsigned grp = __match_any_sync(FULL, hit ? (unsigned)(jj << 1 | (right ? 0 : 1)) : (0x10000u | (unsigned)lane));
            if (hit && (__popc(grp) > 1 || jj == (right ? lastJR : lastJL))) bad = true;
            if (__any_sync(FULL, bad)) { punt = true; break; }
            const unsigned hm = __ballot_sync(FULL, hit);
            if (hm == 0) { __syncwarp(); continue; }
            // the hit reaching furthest extends its side's superstring, the others are checked on the new part
            bool bad2 = false;
#pragma unroll
            for (int side = 0; side < 2; ++side) {
                const bool mine = hit && (right == (side == 0));
                const unsigned ms = __ballot_sync(FULL, mine);
                if (ms == 0) continue;
                u64 *S = side == 0 ? SR : SL;
                const int old = side == 0 ? lenSR : lenSL;
                const unsigned m = __reduce_max_sync(FULL, mine ? ((unsigned)reach << 5 | (unsigned)lane) : 0u);
                const int reachM = (int)(m >> 5), laneM = (int)(m & 31);
                if (reachM > old) {
                    const int sM = __shfl_sync(FULL, s, laneM);
                    const int lo = 32 * lane;
                    if (lane < SS && lo + 32 > old && lo < reachM) {
                        const u64 nb = window_signed(Qs + laneM * SWP, lo - sM);
                        u64 mask = ~0ull;
                        if (old > lo) mask &= ~0ull >> (2 * (old - lo));
                        if (reachM < lo + 32) mask &= ~(~0ull >> (2 * (reachM - lo)));
                        S[lane] = (S[lane] & ~mask) | (nb & mask);
                    }
                    __syncwarp();
                    if (mine && lane != laneM && reach > old) bad2 |= !tail_equal(S, s, Y, max(old - s, 0), len2);
                    if (side == 0) lenSR = reachM; else lenSL = reachM;
                }
                const int lastJ = __shfl_sync(FULL, jj, 31 - __clz(ms));
                if (side == 0) lastJR = lastJ; else lastJL = lastJ;
            }
            if (__any_sync(FULL, bad2)) { punt = true; break; }
            if (hit) {
                const u32 tl = (u32)(type >> 1) << 16 | (u32)len2;
                if (right) { if (jj < myRj) { myRj = jj; myRrid = rid2; myRtl = tl; } }
                else if (jj > myLj) { myLj = jj; myLrid = rid2; myLtl = tl; }
            }
            connections += (u32)__popc(hm);
            __syncwarp();
        }
        __syncwarp();
        if (punt) {         // left to phase_a_kernel (containment marks already made are the ones it makes again)
            if (lane == 0) redo_ids[atomicAdd(redo_count, 1u)] = (u32)i;
            continue;
        }
        // rightExtension = the first right hit (:96-108), leftExtension = the last left hit (:281-357)
        const unsigned rmin = __reduce_min_sync(FULL, (unsigned)myRj << 5 | (unsigned)lane);
        const unsigned lmax = __reduce_max_sync(FULL, (unsigned)(myLj + 1) << 5 | (unsigned)lane);
        const int rl = (int)(rmin & 31), ll = (int)(lmax & 31);
        const int Rj = __shfl_sync(FULL, myRj, rl), Lj = __shfl_sync(FULL, myLj, ll);
        const u32 Rrid = __shfl_sync(FULL, myRrid, rl), Rtl = __shfl_sync(FULL, myRtl, rl);
        const u32 Lrid = __shfl_sync(FULL, myLrid, ll), Ltl = __shfl_sync(FULL, myLtl, ll);
        if (lane == 0) {
            flag5[i] = connections > kConnectionsLimit ? 1 : 0;                       // :443
            extR[i] = Rj != 0x7fffff ? ext_pack(Rrid + 1, Rtl >> 16, (u32)((int)(Rtl & 0xFFFF) - (len1 - Rj))) : ext_pack(0, 0, 0);
            extL[i] = Lj >= 0 ? ext_pack(Lrid + 1, Ltl >> 16, (u32)((int)(Ltl & 0xFFFF) - Lj - P.h)) : ext_pack(0, 0, 0);
        }
        calls += my_calls; probes += my_probes;
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        calls += __shfl_xor_sync(FULL, calls, s);
        probes += __shfl_xor_sync(FULL, probes, s);
    }
    if (lane == 0) { atomicAdd(&counters[0], (unsigned long long)calls); atomicAdd(&counters[1], (unsigned long long)probes); }
}

template <int SW, int MINB>
static void launch_fast_v(Context &c, const SearchParams &P, unsigned long long *d_counters, DevBuf<u32> &redo_ids, DevBuf<unsigned> &redo_n)
{
    constexpr int WARPS = SearchCfg<SW>::WARPS;
    redo_ids.alloc(P.hi - P.lo, c.stream); redo_n.alloc(1, c.stream);
    SG_CUDA(cudaMemsetAsync(redo_n.p, 0, sizeof(unsigned), c.stream));
    const unsigned g = persistent_grid<phase_a_fast_kernel<SW, MINB>>(P.hi - P.lo, WARPS);
    phase_a_fast_kernel<SW, MINB><<<g, WARPS * 32, 0, c.stream>>>(P, c.extR.p, c.extL.p, c.flag5.p, c.cont_max.p, d_counters, redo_ids.p, redo_n.p);
}

// The superstring scan of reads [P.lo, P.hi) (in the order of P.ids when given); the reads it could not certify are
// listed in redo_ids (*redo_n of them; both allocated here).  false: no instantiation for this record stride (long
// reads), nothing launched.
bool launch_phase_a_fast(Context &c, const SearchParams &P, unsigned long long *d_counters, DevBuf<u32> &redo_ids, DevBuf<unsigned> &redo_n)
{
    switch (c.SW) {
        // 4 resident blocks per SM (64 registers): 3 blocks (79 registers) and 5 blocks (48 registers, spills) were measured
        // slower, 12.3 / 11.8 ms against 10.1 ms at cfg2; requesting the home sectors of several window chunks before the
        // first is used was slower too (10.9 / 11.6 / 13.1 ms for 1 / 2 / 3 chunks ahead): the kernel is not short of loads in flight
#define SG_FAST_CASE(SWV) case SWV: launch_fast_v<SWV, 4>(c, P, d_counters, redo_ids, redo_n); break;
        SG_FAST_CASE(2) SG_FAST_CASE(3) SG_FAST_CASE(4) SG_FAST_CASE(5) SG_FAST_CASE(6) SG_FAST_CASE(8)
#undef SG_FAST_CASE
        default: return false;
    }
    SG_LAUNCHED();
    return true;
}

}  // namespace sg
