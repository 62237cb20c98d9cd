// search.cu -- step 3 search kernels (K4 phase A, K5 phase-C candidates).  Restates
// EconomyGraph::buildInitialOverlapGraph phase A (economyGraph/economyGraph.cpp:64-452),
// insertAllEdgesOfRead (:580-638), HashTable::hashTableSearch (hashTable.cpp:193-231) and
// compareStringInBytes[Previous] (economyGraph.cpp:712-808).
//
// One warp per read, three stages per 32 windows:
//   1. PROBE   lane l derives the key of window base+l by funnel shifts from the read's words in shared
//              memory and reads ONE 32-byte sector of the slot index (4 slots).  A 24-bit tag match is
//              taken as "found" (verified in stage 2); a match on a masked key (>= 100 entries) is
//              verified at once through the bucket's first read, exactly like hashTableSearch.
//   2. VERIFY  the (window, bucket entry) pairs of all found windows are flattened into a queue in the
//              reference's order (window ascending, bucket order) and consumed 32 at a time: every
//              lane fetches one partner record in the orientation its entry type asks for and checks
//              the whole overlap by XOR under a mask; the first entry of every bucket also proves the
//              key (a tag collision restarts the read with verified probes).
//   3. EXTEND  the accepted hits of a round feed the unique-extension state machine.  FAST mode checks
//              every hit against the previous hit of its side in parallel (records exchanged through
//              shared memory): as long as no window holds two hits of one side and every adjacent pair
//              is consistent, the reference's chain (economyGraph.cpp:94-437) reduces to "first right
//              hit, last left hit, not ambiguous".  The first round that breaks this converts the
//              state to core.cuh's ExtState and the rest of the read runs the reference's sequential
//              chain hit by hit (EXACT mode) -- still with parallel fetch and verification.
#include <stdlib.h>
#include "search_common.cuh"

namespace sg {

// search_fast.cu
bool launch_phase_a_fast(Context &c, const SearchParams &P, unsigned long long *d_counters, DevBuf<u32> &redo_ids, DevBuf<unsigned> &redo_n);

// FAST-mode scan state of one read (warp-uniform): first right hit, last left hit, last hit of each side
struct FastState {
    u32 Rid = 0, Rtype = 0, Rlen = 0, Lid = 0, Ltype = 0, Llen = 0, connections = 0;
    int cJR = 0, cLenR = 0, firstJR = 0, cJL = 0, cLenL = 0;
};

// X[start+t] == Y[t] for t in [0, ov), ov = min(lenY, lenX-start): X is indexed dynamically (a shared
// memory record with one readable word after it), Y statically (registers or a pointer).  Whole words
// are compared by XOR, the last one under a mask.  `key_bad` = a mismatch under the key masks km0/km1.
template <int SW, typename YT>
__device__ __forceinline__ bool t_overlap_equal(const u64 *X, int lenX, int start, const YT &Y, int lenY, u64 km0, u64 km1,
                                                bool &contained, bool &key_bad)
{
    const int rem = lenX - start;
    contained = lenY <= rem;
    const int ov = contained ? lenY : rem;
    const int wb = ov >> 5;                              // words [0,wb) whole, word wb under bm
    const u64 bm = ~(~0ull >> ((ov & 31) * 2));          // 0 when ov is a multiple of 32
    const int i0 = start >> 5;
    const unsigned s = (unsigned)(start & 31) * 2;
    const bool upper = s >= 32;
    const unsigned s5 = s & 31;
    u64 acc = 0, acck = 0;
    u64 a = X[i0];
#pragma unroll
    for (int w = 0; w < SW; ++w) {
        if (w <= wb) {
            const u64 b = X[i0 + w + 1];
            u64 d = funnel64(a, b, upper, s5) ^ Y[w];
            if (w == wb) d &= bm;
            acc |= d;
            if (w == 0) acck |= d & km0;
            if (w == 1) acck |= d & km1;
            a = b;
        }
    }
    key_bad = acck != 0;
    return acc == 0;
}

// The same test between two records in shared memory, restricted to t in [t0, ov) (bases before t0 are
// known to agree): a real loop over the words that matter instead of SW predicated iterations.
__device__ __forceinline__ bool overlap_equal_from(const u64 *X, int lenX, int start, const u64 *Y, int lenY, int t0)
{
    const int rem = lenX - start;
    const int ov = lenY <= rem ? lenY : rem;
    const int wb = ov >> 5;
    const u64 bm = ~(~0ull >> ((ov & 31) * 2));
    const unsigned s = (unsigned)(start & 31) * 2;
    const bool upper = s >= 32;
    const unsigned s5 = s & 31;
    int w = t0 >> 5;
    const u64 *Xp = X + (start >> 5) + w;
    u64 acc = 0;
    u64 a = Xp[0];
    for (; w < wb; ++w) {
        const u64 b = *++Xp;
        acc |= funnel64(a, b, upper, s5) ^ Y[w];
        a = b;
    }
    acc |= (funnel64(a, Xp[1], upper, s5) ^ Y[w]) & bm;       // w == wb (t0 <= ov)
    return acc == 0;
}

template <int SW>
__device__ __forceinline__ void load_record(const u64 *src, u64 (&q)[SW])
{
#pragma unroll
    for (int w = 0; w < SW; ++w) q[w] = __ldg(&src[w]);
}

// queue item: [32:0] entry (inline) or index into entries | [49:34] window | bit 50 first entry of its
// bucket | bit 51 inline
__device__ __forceinline__ u64 make_item(int jj, bool first, bool inl, u64 payload)
{
    return payload | ((u64)jj << 34) | ((u64)first << 50) | ((u64)inl << 51);
}

// ------------------------------------------------------------------------------------------------
// K4: phase A
// ------------------------------------------------------------------------------------------------
// With an id list P.ids the batch is processed in its order instead of id order (the reads the superstring scan left, or
// the minimizer order that keeps overlapping reads together in time, DESIGN.md section 3); results do not depend on it.
// Registers are cut for 4 resident blocks per SM up to 8 words (3 and 5 were measured slower, DESIGN.md section 3), 1 above.
template <int SW, bool ROUTED>
__global__ void __launch_bounds__(SearchCfg<SW>::WARPS * 32, SW <= 8 ? 4 : 1)
phase_a_kernel(SearchParams P, u64 *__restrict__ extR, u64 *__restrict__ extL, uint8_t *__restrict__ flag5,
               u32 *__restrict__ cont_max, unsigned long long *__restrict__ counters)
{
    constexpr int WARPS = SearchCfg<SW>::WARPS, SWP = SearchCfg<SW>::SWP, SWS = SearchCfg<SW>::SWS, LPI = SearchCfg<SW>::LPI, IPI = 32 / LPI;
    constexpr unsigned FULL = 0xffffffffu;
    __shared__ u64 sXf[WARPS][SW + 1], sXr[WARPS][SW + 1], sPrevR[WARPS][SW + 1], sPrevL[WARPS][SW + 1];   // +1: t_overlap_equal reads one word past
    __shared__ u64 sQ[WARPS][32 * SWP];
    __shared__ u64 sItem[WARPS][32];
    __shared__ ExtState sState[WARPS];
    __shared__ FastState sFast[WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u64 *Xf = sXf[warp], *Xr = sXr[warp], *prevR = sPrevR[warp], *prevL = sPrevL[warp], *Qs = sQ[warp], *items = sItem[warp];
    ExtState &st = sState[warp];
    FastState &fs = sFast[warp];
    const u64 nwarps = (u64)gridDim.x * WARPS;
    const unsigned lt_mask = (1u << lane) - 1u;
    unsigned calls = 0, probes = 0, n_exact = 0, n_restart = 0;      // per warp: far below 2^32
    if (lane == 0) { Xf[SW] = 0; Xr[SW] = 0; prevR[SW] = 0; prevL[SW] = 0; }

    const u64 n_batch = ROUTED ? P.n : (P.n_dev ? (u64)*P.n_dev : P.hi - P.lo);
    for (u64 sb = (u64)blockIdx.x * WARPS + warp; sb < n_batch; sb += nwarps) {
        const u64 i = P.ids ? (u64)P.ids[sb] : P.lo + sb;
        if (lane < SW) { Xf[lane] = P.F[i * SWS + lane]; Xr[lane] = P.RC[i * SWS + lane]; }
        __syncwarp();
        const int len1 = (int)(Xf[SW - 1] & 0xFFFF);
        const int W = len1 - P.h + 1;
        bool exact_probe = false;

    restart:
        // warp-uniform scan state (FAST mode); `exact` switches to the ExtState in shared memory
        // (the FAST-mode values live in shared memory, `fs`, written by lane 0 once per round)
        bool exact = false, hasR = false, hasL = false;
        int curWin = -1;
        unsigned my_calls = 0, my_probes = 0;
        int qn = 0;                                   // items waiting in `items`
        if (lane == 0) fs = FastState();
        __syncwarp();

        for (int base = 0; base < W || qn > 0; base += 32) {
            // ---- stage 1: probe -------------------------------------------------------------------
            u64 payload = 0;
            u32 cnt = 0;
            const int j = base + lane;
            if (ROUTED) {
                bool bad = false;
                if (j < W) {
                    const u64 w = __ldg(&P.wslot[sb * P.wstride + j]);
                    cnt = slot_get_count(w); payload = slot_get_payload(w);
                    if (cnt >= (u32)kHashThreshold) {       // masked key (tag probes only): proven through its
                        if (!P.trusted) {                   // representative, then it reads as absent (hashTable.cpp:203)
                            u64 v0, v1, w0, w1;
                            t_extract_key<SW>(Xf, j, P.h, v0, v1);
                            const u32 ent = (u32)payload;
                            const u64 *X = ((ent & 2) ? P.RC : P.F) + (u64)(ent >> 2) * SWS;
                            const int l = (int)(__ldg(&X[SW - 1]) & 0xFFFF);
                            t_extract_key<SW>(X, (ent & 1) ? l - P.h : 0, P.h, w0, w1);
                            bad = w0 != v0 || w1 != v1;
                        }
                        cnt = 0; payload = 0;
                    }
                }
                if (__any_sync(FULL, bad)) {
                    if (lane == 0) P.redo[sb] = 1;
                    n_restart++;
                    __syncwarp();
                    goto next_read;
                }
            } else if (j < W) {
                u64 v0, v1;
                t_extract_key<SW>(Xf, j, P.h, v0, v1);
                probe_window<SW>(P, v0, v1, exact_probe, payload, cnt);
            }
            u32 incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const u32 y = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += y; }
            const int T = (int)__shfl_sync(FULL, incl, 31);
            const bool last_chunk = base + 32 >= W;
            int consumed = 0;

            // ---- stage 2 + 3: rounds of 32 items ------------------------------------------------------
            for (;;) {
                const int avail = qn + (T - consumed);
                if (avail == 0 || (avail < 32 && !last_chunk)) break;
                const int take = avail < 32 ? avail : 32;
                // lanes [0,qn) take queued items, lanes [qn,take) items consumed.. of this chunk
                u64 item = 0;
                {
                    int t = consumed + lane - qn;
                    const bool from_chunk = lane >= qn && lane < take;
                    if (t < 0) t = 0;
                    if (t >= T) t = T > 0 ? T - 1 : 0;
                    int lo = 0;
#pragma unroll
                    for (int step = 16; step > 0; step >>= 1) {
                        const u32 pm = __shfl_sync(FULL, incl, lo + step - 1);
                        if (pm <= (u32)t) lo += step;
                    }
                    if (lo > 31) lo = 31;
                    const u32 ex = __shfl_sync(FULL, incl - cnt, lo);
                    const u32 c = __shfl_sync(FULL, cnt, lo);
                    const u64 pay = __shfl_sync(FULL, payload, lo);
                    const u32 e = (u32)t - ex;
                    if (from_chunk) item = make_item(base + lo, e == 0, c == 1, c == 1 ? pay : pay + e);
                    else if (lane < qn) item = items[lane];
                }
                consumed += take - qn;
                qn = 0;
                const bool valid = lane < take;

                // ---- verify ---------------------------------------------------------------------------
                const int jj = (int)((item >> 34) & 0xFFFF);
                const bool first = (item >> 50) & 1, inl = (item >> 51) & 1;
                bool hit = false, right = false, fp = false, need = false, load = false;
                u32 rid2 = 0;
                int len2 = 0, type = 0;
                const u64 *rec = P.F;
                if (valid) {
                    const u32 ent = inl ? (u32)(item & 0xFFFFFFFFull) : __ldg(&P.entries[item & 0x1FFFFFFFFull]);
                    rid2 = ent >> 2; type = (int)(ent & 3);
                    right = !(type & 1);
                    need = rid2 != (u32)i && (right ? gate_right(jj, len1, P.k) : gate_left(jj, P.k, P.h));
                    load = need || first;
                    rec = (partner_uses_rc(type) ? P.RC : P.F) + (u64)rid2 * SWS;
                }
                // partner records -> shared memory, LPI lanes per record with one 256-bit load each: one memory
                // request per record, however many sectors it spans
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
                if (load) {
                    const u64 *Y = Qs + lane * SWP;
                    len2 = (int)(Y[SW - 1] & 0xFFFF);
                    bool contained, key_bad;
                    u64 km0, km1;
                    key_masks(P.h, km0, km1);
                    const bool ok = t_overlap_equal<SW>(right ? Xf : Xr, len1, right ? jj : len1 - jj - P.h, Y, len2, km0, km1, contained, key_bad);
                    fp = first && key_bad;
                    if (need) {
                        my_calls++;
                        if (ok && contained) atomicMax(&cont_max[rid2], (u32)(i + 1));      // economyGraph.cpp:735
                        hit = ok && !contained;
                    }
                }
                if (__any_sync(FULL, fp)) {          // tag collision: redo this read with verified probes
                    n_restart++;
                    __syncwarp();
                    if (ROUTED) { if (lane == 0) P.redo[sb] = 1; goto next_read; }
                    exact_probe = true;
                    goto restart;
                }
                unsigned hm = __ballot_sync(FULL, hit);
                if (hm == 0) { __syncwarp(); continue; }

                // ---- extend -------------------------------------------------------------------------
                if (!exact) {
                    const unsigned mR = __ballot_sync(FULL, hit && right), mL = hm & ~mR;
                    const unsigned lower = (right ? mR : mL) & lt_mask;
                    const int src = lower ? 31 - __clz(lower) : -1;
                    const int pj = __shfl_sync(FULL, jj, src < 0 ? lane : src);
                    const int plen = __shfl_sync(FULL, len2, src < 0 ? lane : src);
                    bool anomaly = false;
                    if (hit) {
                        const u64 *prec = nullptr;
                        int prevJ = 0, prevLen = 0;
                        if (src >= 0) { prec = Qs + src * SWP; prevJ = pj; prevLen = plen; }
                        else if (right ? hasR : hasL) { prec = right ? prevR : prevL; prevJ = right ? fs.cJR : fs.cJL; prevLen = right ? fs.cLenR : fs.cLenL; }
                        if (prec) {
                            // Both records agree with read i over its span (verified above), so only the bases past
                            // read i's end can differ: right, Q[t] with t >= len1 - jj; left (records are oriented like
                            // revcomp(read i)), prev[t] with t >= prevJ + h.
                            const u64 *mine = Qs + lane * SWP;
                            if (prevJ == jj) anomaly = true;                      // two hits of one side in one window
                            else if (right) anomaly = !overlap_equal_from(prec, prevLen, jj - prevJ, mine, len2, len1 - jj);   // :110-112
                            else anomaly = !overlap_equal_from(mine, len2, jj - prevJ, prec, prevLen, prevJ + P.h);           // :295-297
                        }
                    }
                    if (!__any_sync(FULL, anomaly)) {
                        __syncwarp();
                        if (mR) {
                            if (!hasR) {      // rightExtension = the first right hit (longest overlap), :96-108
                                const int f = __ffs(mR) - 1;
                                const int jf = __shfl_sync(FULL, jj, f), lf = __shfl_sync(FULL, len2, f);
                                const u32 rf = __shfl_sync(FULL, rid2, f);
                                const int tf = __shfl_sync(FULL, type, f);
                                if (lane == 0) { fs.Rid = rf + 1; fs.Rtype = (u32)(tf >> 1); fs.Rlen = (u32)(lf - (len1 - jf)); fs.firstJR = jf; }
                                hasR = true;
                            }
                            const int l = 31 - __clz(mR);
                            const int jl = __shfl_sync(FULL, jj, l), ll = __shfl_sync(FULL, len2, l);
                            if (lane == 0) { fs.cJR = jl; fs.cLenR = ll; }
                            if (lane < SW) prevR[lane] = Qs[l * SWP + lane];
                        }
                        if (mL) {             // leftExtension = the last left hit (longest overlap), :281-357
                            const int l = 31 - __clz(mL);
                            const int jl = __shfl_sync(FULL, jj, l), ll = __shfl_sync(FULL, len2, l);
                            const u32 rl = __shfl_sync(FULL, rid2, l);
                            const int tl = __shfl_sync(FULL, type, l);
                            if (lane == 0) { fs.cJL = jl; fs.cLenL = ll; fs.Lid = rl + 1; fs.Ltype = (u32)(tl >> 1); fs.Llen = (u32)(ll - jl - P.h); }
                            hasL = true;
                            if (lane < SW) prevL[lane] = Qs[l * SWP + lane];
                        }
                        if (lane == 0) fs.connections += (u32)__popc(hm);
                        __syncwarp();
                        continue;
                    }
                    // convert to the reference's sequential state as of just before this round
                    exact = true;
                    n_exact++;
                    curWin = __shfl_sync(FULL, jj, __ffs(hm) - 1);
                    if (lane == 0) {
                        ext_init(st);
                        st.Rid = fs.Rid; st.Rtype = fs.Rtype; st.Rlen = fs.Rlen; st.Lid = fs.Lid; st.Ltype = fs.Ltype; st.Llen = fs.Llen;
                        st.prevJR = fs.cJR; st.prevLenR = fs.cLenR; st.prevPL = len1 - fs.cJL - P.h; st.prevLenL = fs.cLenL;
                        st.markAmbigR = (hasR && fs.cJR == curWin) ? 1 : 0;
                        st.markFirstR = (hasR && fs.firstJR == curWin) ? 1 : 0;
                        st.markAmbigL = (hasL && fs.cJL == curWin) ? 1 : 0;
                        st.connections = fs.connections;
                    }
                    __syncwarp();
                }
                while (hm) {
                    const int b = __ffs(hm) - 1;
                    hm &= hm - 1;
                    const int jb = __shfl_sync(FULL, jj, b);
                    if (jb != curWin) { curWin = jb; if (lane == 0) ext_new_window(st); }      // :86-88
                    __syncwarp();
                    if (lane == b) {
                        if (right) ext_right_hit(st, prevR, Qs + lane * SWP, SW, rid2 + 1, type >> 1, jj, len1, len2);
                        else ext_left_hit(st, prevL, Qs + lane * SWP, SW, rid2 + 1, type >> 1, jj, P.h, len1, len2);
                    }
                    __syncwarp();
                }
            }
            // leftover items of this chunk wait for the next one
            {
                const int rem = T - consumed;      // < 32 - qn
                int t = consumed + lane;
                const bool mine = lane < rem;
                if (t >= T) t = T > 0 ? T - 1 : 0;
                int lo = 0;
#pragma unroll
                for (int step = 16; step > 0; step >>= 1) {
                    const u32 pm = __shfl_sync(FULL, incl, lo + step - 1);
                    if (pm <= (u32)t) lo += step;
                }
                if (lo > 31) lo = 31;
                const u32 ex = __shfl_sync(FULL, incl - cnt, lo);
                const u32 c = __shfl_sync(FULL, cnt, lo);
                const u64 pay = __shfl_sync(FULL, payload, lo);
                const u32 e = (u32)t - ex;
                if (mine) items[qn + lane] = make_item(base + lo, e == 0, c == 1, c == 1 ? pay : pay + e);
                qn += rem;
                __syncwarp();
            }
            my_probes += (j < W);
        }
        __syncwarp();
        if (lane == 0) {
            if (exact) {
                flag5[i] = st.connections > kConnectionsLimit ? 1 : 0;              // :443
                const bool amb = st.itsAmbigR == 1 || st.itsAmbigL == 1;           // :446-450
                extR[i] = ext_pack(st.Rid, st.Rtype, amb ? 0u : st.Rlen);
                extL[i] = ext_pack(st.Lid, st.Ltype, amb ? 0u : st.Llen);
            } else {
                flag5[i] = fs.connections > kConnectionsLimit ? 1 : 0;
                extR[i] = ext_pack(fs.Rid, fs.Rtype, fs.Rlen);
                extL[i] = ext_pack(fs.Lid, fs.Ltype, fs.Llen);
            }
        }
        calls += my_calls; probes += my_probes;
    next_read:
        __syncwarp();
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        calls += __shfl_xor_sync(FULL, calls, s);
        probes += __shfl_xor_sync(FULL, probes, s);
    }
    if (lane == 0) {
        atomicAdd(&counters[0], (unsigned long long)calls); atomicAdd(&counters[1], (unsigned long long)probes);
        if (n_exact) atomicAdd(&counters[2], (unsigned long long)n_exact);
        if (n_restart) atomicAdd(&counters[3], (unsigned long long)n_restart);
    }
}

// ------------------------------------------------------------------------------------------------
// K5: phase-C candidates.  For every read r1 still unexplored after phase B (state 0) list, in the
// reference's order, every (read2, edge type, overhang) insertAllEdgesOfRead would test positive
// (economyGraph.cpp:599-631), restricted to read2 that are themselves state 0 (any other state is
// skipped at :605 and never returns to 0).  Pass 1 counts, pass 2 fills.
// candidate = read2(1-based) << 32 | edgeType << 20 | (overhang & 0xFFFFF)
// ------------------------------------------------------------------------------------------------
template <int SW, bool FILL, bool ROUTED>
__global__ void __launch_bounds__(SearchCfg<SW>::WARPS * 32)
phase_c_kernel(SearchParams P, const u32 *__restrict__ s_ids, u64 nS, const uint8_t *__restrict__ explored,
               u32 *__restrict__ counts, const u32 *__restrict__ offsets, u64 *__restrict__ cand)
{
    constexpr int WARPS = SearchCfg<SW>::WARPS;
    __shared__ u64 sXf[WARPS][SW + 1], sXr[WARPS][SW + 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u64 *Xf = sXf[warp], *Xr = sXr[warp];
    if (lane == 0) { Xf[SW] = 0; Xr[SW] = 0; }
    const u64 nwarps = (u64)gridDim.x * WARPS;
    for (u64 s = (u64)blockIdx.x * WARPS + warp; s < nS; s += nwarps) {
        const u64 i = s_ids[s];      // 0-based
        if (lane < SW) { Xf[lane] = P.F[i * SearchCfg<SW>::SWS + lane]; Xr[lane] = P.RC[i * SearchCfg<SW>::SWS + lane]; }
        __syncwarp();
        const int len1 = (int)(Xf[SW - 1] & 0xFFFF);
        const int W = len1 - P.h + 1;
        u32 total = 0;
        const u64 out_base = FILL ? offsets[s] : 0;
        for (int base = 0; base < W; base += 32) {
            const int j = base + lane;
            u64 payload = 0;
            u32 cnt = 0;
            if (ROUTED) {          // verified answers of the owning shards, s_ids is the routed batch
                if (j < W) {
                    const u64 w = __ldg(&P.wslot[s * P.wstride + j]);
                    cnt = slot_get_count(w); payload = slot_get_payload(w);
                }
            } else if (j < W) {
                u64 v0, v1;
                t_extract_key<SW>(Xf, j, P.h, v0, v1);
                probe_window<SW>(P, v0, v1, true, payload, cnt);
            }
            unsigned fm = __ballot_sync(0xffffffffu, cnt != 0);
            while (fm) {
                const int l = __ffs(fm) - 1;
                fm &= fm - 1;
                const int jj = base + l;
                const u64 pay = __shfl_sync(0xffffffffu, payload, l);
                const u32 c = __shfl_sync(0xffffffffu, cnt, l);
                const bool gateR = gate_right(jj, len1, P.k), gateL = gate_left(jj, P.k, P.h);
                for (u32 e0 = 0; e0 < c; e0 += 32) {
                    const u32 e = e0 + lane;
                    bool ok = false;
                    u64 rec = 0;
                    if (e < c) {
                        const u32 ent = c == 1 ? (u32)pay : __ldg(&P.entries[pay + e]);
                        const u32 rid2 = ent >> 2;
                        const int type = (int)(ent & 3);
                        const bool right = !(type & 1);
                        if (rid2 != (u32)i && explored[rid2] == 0 && (right ? gateR : gateL)) {
                            u64 q[SW];
                            load_record<SW>((partner_uses_rc(type) ? P.RC : P.F) + (u64)rid2 * SearchCfg<SW>::SWS, q);
                            const int len2 = (int)(q[SW - 1] & 0xFFFF);
                            bool contained, kb;
                            ok = t_overlap_equal<SW>(right ? Xf : Xr, len1, right ? jj : len1 - jj - P.h, q, len2, 0ull, 0ull, contained, kb);
                            rec = candidate_record(type, jj, P.h, len1, len2, rid2);
                        }
                    }
                    const unsigned om = __ballot_sync(0xffffffffu, ok);
                    if (FILL && ok) cand[out_base + total + __popc(om & ((1u << lane) - 1u))] = rec;
                    total += __popc(om);
                }
            }
        }
        if (!FILL && lane == 0) counts[s] = total;
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
// the local search of a slice and its redo pass after the scan, or (ROUTED) one routed batch; the grid covers the whole
// slice or batch even when only the device knows how many ids a list holds
template <int SW, bool ROUTED>
static void launch_phase_a(Context &c, const SearchParams &P, unsigned long long *d_counters)
{
    constexpr int WARPS = SearchCfg<SW>::WARPS;
    const unsigned g = persistent_grid<phase_a_kernel<SW, ROUTED>>(ROUTED ? P.n : P.hi - P.lo, WARPS);
    phase_a_kernel<SW, ROUTED><<<g, WARPS * 32, 0, c.stream>>>(P, c.extR.p, c.extL.p, c.flag5.p, c.cont_max.p, d_counters);
}

#define SG_DISPATCH_SW(SWV, CALL)                                                       \
    switch (SWV) {                                                                      \
        case 2: { constexpr int SWC = 2; CALL; } break;                                 \
        case 3: { constexpr int SWC = 3; CALL; } break;                                 \
        case 4: { constexpr int SWC = 4; CALL; } break;                                 \
        case 5: { constexpr int SWC = 5; CALL; } break;                                 \
        case 6: { constexpr int SWC = 6; CALL; } break;                                 \
        case 8: { constexpr int SWC = 8; CALL; } break;                                 \
        case 12: { constexpr int SWC = 12; CALL; } break;                               \
        case 16: { constexpr int SWC = 16; CALL; } break;                               \
        case 32: { constexpr int SWC = 32; CALL; } break;                               \
        default: throw CudaError("unsupported record stride");                         \
    }

// ---- read schedule (read_order = 1): reads sorted by their minimizer, so that reads sharing bases are searched together ----
// The key of a read is the least hash over its 32-base words (m = 32: one u64, cut out by a constant funnel shift); the
// hash is one 64-bit multiply, top 32 bits.  Forward words only: canonical words (the smaller of a word and its reverse
// complement) gave the same search time at cfg4 and cost 3.4 times as much to compute (DESIGN.md section 3).
constexpr u64 kMinimizerMul = 0x9e3779b97f4a7c15ull;

// One thread per read: a warp loads its 32 consecutive records with coalesced loads into shared memory (rows padded to
// an odd stride), then every lane scans its own record.
template <int SW>
__global__ void __launch_bounds__((SearchCfg<SW>::SWS <= 16 ? 8 : 4) * 32)
minimizer_kernel(const u64 *__restrict__ F, u64 lo, u64 n, u64 *__restrict__ key, u32 *__restrict__ id)
{
    constexpr int SWS = SearchCfg<SW>::SWS, ROW = SWS + 1, WARPS = SWS <= 16 ? 8 : 4;
    __shared__ u64 sX[WARPS][32 * ROW];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u64 *X = sX[warp];
    const u64 ngroups = (n + 31) / 32, nwarps = (u64)gridDim.x * WARPS;
    for (u64 g = (u64)blockIdx.x * WARPS + warp; g < ngroups; g += nwarps) {
        const u64 s0 = g * 32;
        const int nr = n - s0 < 32 ? (int)(n - s0) : 32;
        const u64 *src = F + (lo + s0) * SWS;
        __syncwarp();
#pragma unroll
        for (int t = 0; t < SWS; ++t) {
            const int k = 32 * t + lane, r = k / SWS, w = k % SWS;
            if (r < nr) X[r * ROW + w] = __ldg(&src[k]);
        }
        __syncwarp();
        if (lane < nr) {
            const u64 *x = X + lane * ROW;
            const int last = (int)(x[SW - 1] & 0xFFFF) - 32;      // start of the last whole word of the read
            u32 m = 0xFFFFFFFFu;
#pragma unroll(SW <= 8 ? SW : 1)
            for (int w = 0; w < SW; ++w) {
                const u64 a = x[w], b = x[w + 1];                 // x[SW]: storage or row padding, masked off below
#pragma unroll
                for (int sh = 0; sh < 32; ++sh) {
                    const u64 win = sh == 0 ? a : ((a << (2 * sh)) | (b >> (64 - 2 * sh)));
                    const u32 hv = (u32)((win * kMinimizerMul) >> 32);
                    m = (32 * w + sh <= last && hv < m) ? hv : m;
                }
            }
            key[s0 + lane] = m;
            id[s0 + lane] = (u32)(lo + s0 + lane);
        }
    }
}

// ids of [lo, hi) in minimizer order (device array owned by the caller's arena scope).  The sort is stable: reads with
// one key keep id order.
template <int SW>
static void launch_minimizer(Context &c, u64 lo, u64 n, u64 *key, u32 *id)
{
    constexpr int WARPS = SearchCfg<SW>::SWS <= 16 ? 8 : 4;
    u64 g = (n + 32 * WARPS - 1) / (32 * WARPS);
    if (g > (u64)kSMs * 16) g = (u64)kSMs * 16;
    minimizer_kernel<SW><<<(unsigned)g, WARPS * 32, 0, c.stream>>>(c.F.p, lo, n, key, id);
}

static const u32 *minimizer_order(Context &c, u64 lo, u64 hi, DevBuf<u64> &ka, DevBuf<u64> &kb, DevBuf<u32> &va, DevBuf<u32> &vb)
{
    cudaStream_t st = c.stream;
    const u64 n = hi - lo;
    ka.alloc(n, st); kb.alloc(n, st); va.alloc(n, st); vb.alloc(n, st);
    SG_DISPATCH_SW(c.SW, launch_minimizer<SWC>(c, lo, n, ka.p, va.p));
    SG_LAUNCHED();
    SortCols cols;
    cols.a[0] = ka.p; cols.a[1] = kb.p; cols.b[0] = cols.b[1] = nullptr; cols.v[0] = va.p; cols.v[1] = vb.p;
    const int cur = radix_sort_bits(cols, 0, n, false, 0, 32, st);
    return cols.v[cur];
}

template <int SW>
static void launch_phase_c(Context &c, const SearchParams &P, const u32 *s_ids, u64 nS, u32 *counts, const u32 *offsets, u64 *cand, bool fill)
{
    constexpr int WARPS = SearchCfg<SW>::WARPS;
    const unsigned g = search_grid(nS, WARPS, 8);
    if (P.wslot) {
        if (fill) phase_c_kernel<SW, true, true><<<g, WARPS * 32, 0, c.stream>>>(P, s_ids, nS, c.explored.p, counts, offsets, cand);
        else phase_c_kernel<SW, false, true><<<g, WARPS * 32, 0, c.stream>>>(P, s_ids, nS, c.explored.p, counts, offsets, cand);
    } else {
        if (fill) phase_c_kernel<SW, true, false><<<g, WARPS * 32, 0, c.stream>>>(P, s_ids, nS, c.explored.p, counts, offsets, cand);
        else phase_c_kernel<SW, false, false><<<g, WARPS * 32, 0, c.stream>>>(P, s_ids, nS, c.explored.p, counts, offsets, cand);
    }
}

// Default schedule: the minimizer order pays once the records and the slot index the search reads at random are far
// larger than L2 (cfg4, 4.9 GB: faster in that order; cfg2, 0.4 GB: slower, DESIGN.md section 3).
constexpr u64 kReadOrderMinBytes = (u64)1 << 30;

static bool read_order_pays(const Context &c)
{
    const u64 bytes = 2 * c.cnt.unique_reads * (u64)c.SWS * sizeof(u64) + c.cap * sizeof(u64);
    return bytes >= kReadOrderMinBytes;
}

static SearchParams make_params(const Context &c)
{
    SearchParams P;
    P.F = c.F.p; P.RC = c.RC.p; P.slots = c.slots.p; P.entries = c.entries.p;
    P.shards = c.tb_shards > 1 ? c.tb_shards : 1;
    P.nsec = c.cap / kSlotsPerSector / (u64)P.shards; P.U = c.cnt.unique_reads; P.lo = 0; P.hi = P.U; P.h = c.h; P.k = c.min_overlap;
    P.wslot = nullptr; P.ids = nullptr; P.redo = nullptr; P.n = 0; P.wstride = 0; P.trusted = 0; P.n_dev = nullptr;
    return P;
}

// the answers of the routed batch (shard.cu) instead of the local table
static void use_routed_batch(const Context &c, SearchParams &P)
{
    P.slots = nullptr; P.nsec = 0;
    P.wslot = c.rt_wslot.p; P.entries = c.rt_entries_view; P.wstride = c.rt_wstride; P.n = c.rt_n;
    P.ids = c.rt_is_list ? c.rt_ids.p : nullptr; P.lo = c.rt_first; P.hi = c.rt_first + c.rt_n;
    P.trusted = c.rt_exact ? 1 : 0;
}

// Rank `rank`'s slice [lo, hi) of the reads cut into `world` equal chunks, and the phase-A arrays of all chunks (the
// exchange moves whole chunks); cont_max and the counters start at 0.
static void begin_phase_a(Context &c, int rank, int world, u64 &lo, u64 &hi)
{
    cudaStream_t st = c.stream;
    SG_CHECK(world >= 1 && rank >= 0 && rank < world, "bad rank / world");
    const u64 U = c.cnt.unique_reads;
    const u64 chunk = partition_chunk(U, world), padded = chunk * (u64)world;
    c.pa_chunk = chunk; c.pa_world = world;
    lo = (u64)rank * chunk < U ? (u64)rank * chunk : U;
    hi = lo + chunk < U ? lo + chunk : U;
    c.have_phase_a = false; c.have_phase_b = false; c.have_graph = false;
    c.extR.alloc(padded, st); c.extL.alloc(padded, st); c.flag5.alloc(padded, st); c.cont_max.alloc(padded, st);
    c.cnt.compare_calls = 0; c.cnt.window_probes = 0; c.cnt.slow_path_reads = 0; c.cnt.probe_restarts = 0;
    if (U > 0) SG_CUDA(cudaMemsetAsync(c.cont_max.p, 0, padded * sizeof(u32), st));
}

// The phase-A kernels' counters (compare calls, window probes, slow-path reads, probe restarts), zeroed, and the time of
// the launches between construction and finish().
struct PhaseARun {
    cudaStream_t st;
    DevBuf<unsigned long long> counters;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    explicit PhaseARun(cudaStream_t s) : st(s), counters(4, s)
    {
        SG_CUDA(cudaMemsetAsync(counters.p, 0, 4 * sizeof(unsigned long long), st));
        SG_CUDA(cudaEventCreate(&e0)); SG_CUDA(cudaEventCreate(&e1));
        SG_CUDA(cudaEventRecord(e0, st));
    }
    ~PhaseARun() { cudaEventDestroy(e0); cudaEventDestroy(e1); }
    // waits for the launches; h = the counters, returns their time in ms
    float finish(unsigned long long (&h)[4])
    {
        SG_CUDA(cudaEventRecord(e1, st));
        SG_CUDA(cudaMemcpyAsync(h, counters.p, sizeof(h), cudaMemcpyDeviceToHost, st));
        SG_CUDA(cudaStreamSynchronize(st));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        return ms;
    }
};

void stage_phase_a(Context &c, int rank, int world)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    SG_CHECK(c.have_table, "build_hash_table must run before the overlap search");
    SG_CHECK(c.tb_world == 1, "this context holds one shard of the table: use the routed search (sage2gpu_route_*)");
    SearchParams P = make_params(c);
    begin_phase_a(c, rank, world, P.lo, P.hi);
    if (c.cnt.unique_reads == 0) { c.have_phase_a = true; return; }
    if (world > 1) {      // slices of other ranks (and the padding) are defined before the exchange overwrites them
        const u64 padded = c.pa_chunk * (u64)world;
        SG_CUDA(cudaMemsetAsync(c.extR.p, 0, padded * sizeof(u64), st));
        SG_CUDA(cudaMemsetAsync(c.extL.p, 0, padded * sizeof(u64), st));
        SG_CUDA(cudaMemsetAsync(c.flag5.p, 0, padded, st));
    }
    // SAGE2GPU_READ_ORDER=id|minimizer ("minhash" is read as minimizer); unset: by footprint
    static const int env_order = [] { const char *e = getenv("SAGE2GPU_READ_ORDER"); return !e ? -1 : (e[0] == 'm' ? 1 : 0); }();
    static const bool env_fast = [] { const char *e = getenv("SAGE2GPU_PA_FAST"); return !(e && e[0] == '0'); }();
    const int order = c.opt_read_order >= 0 ? c.opt_read_order : env_order;
    const bool by_minimizer = order >= 0 ? order == 1 : read_order_pays(c);
    const bool fast = c.opt_fast_scan < 0 ? env_fast : c.opt_fast_scan == 1;
    DevBuf<u64> oka, okb;
    DevBuf<u32> ova, ovb, redo_ids;
    DevBuf<unsigned> redo_n;
    // schedule that keeps overlapping reads together in time (DESIGN.md section 3); the ordering is part of the stage's
    // time, not of the search kernel's
    if (P.hi > P.lo && by_minimizer) P.ids = minimizer_order(c, P.lo, P.hi, oka, okb, ova, ovb);
    PhaseARun run(st);
    if (P.hi > P.lo) {
        // the superstring scan first (search_fast.cu); the general kernel then takes the reads it could not certify
        if (fast && launch_phase_a_fast(c, P, run.counters.p, redo_ids, redo_n)) { P.ids = redo_ids.p; P.n_dev = redo_n.p; }
        SG_DISPATCH_SW(c.SW, (launch_phase_a<SWC, false>(c, P, run.counters.p)));
        SG_LAUNCHED();
    }
    unsigned long long h[4];
    c.tm.phase_a_kernel = run.finish(h);
    c.cnt.compare_calls = h[0];
    c.cnt.window_probes = h[1];
    c.cnt.slow_path_reads = h[2];
    c.cnt.probe_restarts = h[3];
    c.cnt.fast_path_reads = 0;
    if (redo_n.p) {
        unsigned nr = 0;
        SG_CUDA(cudaMemcpyAsync(&nr, redo_n.p, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
        SG_CUDA(cudaStreamSynchronize(st));
        c.cnt.fast_path_reads = (P.hi - P.lo) - nr;
    }
    c.have_phase_a = true;
}

// ---- single-process multi-GPU host: the phase-A arrays of rank src_rank's slice come over from its context -------------
__global__ void __launch_bounds__(256) max_merge_kernel(u32 *__restrict__ dst, const u32 *__restrict__ src, u64 n)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) { const u32 v = src[i]; if (v > dst[i]) dst[i] = v; }
}

void stage_phase_a_import(Context &c, Context &src, int src_rank)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    SG_CHECK(c.have_phase_a && src.have_phase_a && c.pa_chunk == src.pa_chunk && c.pa_world == src.pa_world, "both contexts must have searched slices of the same partition");
    SG_CHECK(src_rank >= 0 && src_rank < c.pa_world, "bad source rank");
    const u64 chunk = c.pa_chunk, off = (u64)src_rank * chunk, padded = chunk * (u64)c.pa_world;
    if (chunk == 0) return;
    SG_CUDA(cudaMemcpyPeerAsync(c.extR.p + off, c.device, src.extR.p + off, src.device, chunk * sizeof(u64), st));
    SG_CUDA(cudaMemcpyPeerAsync(c.extL.p + off, c.device, src.extL.p + off, src.device, chunk * sizeof(u64), st));
    SG_CUDA(cudaMemcpyPeerAsync(c.flag5.p + off, c.device, src.flag5.p + off, src.device, chunk, st));
    // economyGraph.cpp:735 -- the largest id that found the read contained: element-wise maximum over the ranks' arrays
    DevBuf<u32> tmp(padded, st);
    SG_CUDA(cudaMemcpyPeerAsync(tmp.p, c.device, src.cont_max.p, src.device, padded * sizeof(u32), st));
    unsigned g = grid_for(padded, 256, 4);
    if (g > kSMs * 16u) g = kSMs * 16u;
    max_merge_kernel<<<g, 256, 0, st>>>(c.cont_max.p, tmp.p, padded);
    SG_LAUNCHED();
    SG_CUDA(cudaStreamSynchronize(st));
}

// ---- phase A over a sharded table: begin (allocate the slice's arrays) / one routed batch / end ------------------
void stage_phase_a_sharded_begin(Context &c, int rank, int world)
{
    cudaStream_t st = c.stream;
    SG_CHECK(c.have_table, "build_hash_table[_shard] must run before the overlap search");
    begin_phase_a(c, rank, world, c.pa_lo, c.pa_hi);
    c.rt_redo.alloc(c.pa_chunk, st);
    c.tm.phase_a_kernel = 0;
    if (c.cnt.unique_reads == 0) return;
    const u64 padded = c.pa_chunk * (u64)world;
    SG_CUDA(cudaMemsetAsync(c.extR.p, 0, padded * sizeof(u64), st));
    SG_CUDA(cudaMemsetAsync(c.extL.p, 0, padded * sizeof(u64), st));
    SG_CUDA(cudaMemsetAsync(c.flag5.p, 0, padded, st));
    SG_CUDA(cudaMemsetAsync(c.rt_redo.p, 0, c.pa_chunk, st));
}

// K4 on the routed batch (route_begin .. route_finish); returns the reads of the batch flagged for the redo pass
u64 stage_phase_a_routed(Context &c)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    SG_CHECK(c.rt_state == 2, "route_finish must precede the routed search");
    SG_CHECK(c.rt_what == 0 || c.rt_what == 2, "the routed batch is not a phase-A batch");
    c.rt_state = 0;
    if (c.rt_n == 0) return 0;
    SearchParams P = make_params(c);
    use_routed_batch(c, P);
    // redo flags: by position in the slice for range batches; a private array for the redo list itself
    DevBuf<uint8_t> redo2;
    if (c.rt_is_list) { redo2.alloc(c.rt_n, st); SG_CUDA(cudaMemsetAsync(redo2.p, 0, c.rt_n, st)); P.redo = redo2.p; }
    else P.redo = c.rt_redo.p + (c.rt_first - c.pa_lo);
    PhaseARun run(st);
    SG_DISPATCH_SW(c.SW, (launch_phase_a<SWC, true>(c, P, run.counters.p)));
    SG_LAUNCHED();
    unsigned long long h[4];
    const float ms = run.finish(h);
    c.cnt.compare_calls += h[0];
    c.cnt.window_probes += h[1];
    c.cnt.slow_path_reads += h[2];
    if (!c.rt_exact) c.cnt.probe_restarts += h[3];
    else SG_CHECK(h[3] == 0, "a verified answer failed its proof in the search kernel");
    c.tm.phase_a_kernel += ms;
    return h[3];
}

void stage_phase_a_sharded_end(Context &c)
{
    c.have_phase_a = true;
}

// used by graph.cu
void launch_phase_c_candidates(Context &c, const u32 *s_ids, u64 nS, u32 *counts, const u32 *offsets, u64 *cand, bool fill)
{
    SearchParams P = make_params(c);
    if (c.tb_world > 1 || c.rt_for_c) {      // sharded table: the state-0 reads were routed (what = 1) before finish_graph
        SG_CHECK(c.rt_for_c && c.rt_n == nS, "the reads left for phase C must be routed before finish_graph");
        use_routed_batch(c, P);
    }
    SG_DISPATCH_SW(c.SW, launch_phase_c<SWC>(c, P, s_ids, nS, counts, offsets, cand, fill));
    SG_LAUNCHED();
}

}  // namespace sg
