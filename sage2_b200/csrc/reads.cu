// reads.cu -- step 1 on device: filter + canonicalise + 2-bit pack (K1), sort + dedupe with
// frequencies + packed reverse complements (K2).  Restates ReadLoader::readDatasetInBytes /
// insertReadIntoList / organizeReads (inputReader/readLoader.cpp:133-260) and the utils.cpp helpers
// they call (isGoodRead :144, reverseComplement :73, charsToBytes :96).
#include <stdlib.h>
#include "context.h"

namespace sg {

// ------------------------------------------------------------------------------------------------
// K1: one warp per read.  Lane l of round w handles base 32w+l, so one round assembles exactly one
// 64-bit record word of the read and one of its reverse complement (two __reduce_or_sync each).
// Bad reads (length <= k, non-ACGT, utils.cpp:144-166) become all-ones records that sort last.
// ------------------------------------------------------------------------------------------------
constexpr int K1_WARPS = 8;

__global__ void __launch_bounds__(K1_WARPS * 32) max_len_kernel(const int64_t *__restrict__ off, u64 n, int *out)
{
    int m = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const int64_t d = off[i + 1] - off[i];
        const int l = d > 0x7FFFFFFF ? 0x7FFFFFFF : (int)d;
        m = l > m ? l : m;
    }
    m = __reduce_max_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

__global__ void __launch_bounds__(K1_WARPS * 32) pack_kernel(const uint8_t *__restrict__ bases, const int64_t *__restrict__ off,
                                                              u64 n, int k, int SW, u64 *__restrict__ rec,
                                                              unsigned long long *counters /*[0]=good,[1]=bp*/)
{
    // per warp: the read's characters (coalesced byte loads, zero padded to a multiple of 128), its packed
    // forward words (written byte-wise, most significant byte first) and its reverse complement
    __shared__ __align__(16) uint8_t sB[K1_WARPS][32 * kMaxWords];
    __shared__ u64 sF[K1_WARPS][kMaxWords], sR[K1_WARPS][kMaxWords];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u64 nwarps = (u64)gridDim.x * K1_WARPS;
    unsigned long long good = 0, bp = 0;
    uint8_t *B = sB[warp];
    uint8_t *Fb = reinterpret_cast<uint8_t *>(sF[warp]);
    for (u64 r = (u64)blockIdx.x * K1_WARPS + warp; r < n; r += nwarps) {
        const int64_t o = off[r];
        const int64_t len64 = off[r + 1] - o;
        const int max_ok = 32 * SW - 8;
        bool bad = len64 <= (int64_t)k || len64 > (int64_t)max_ok;
        const int len = bad ? 0 : (int)len64;
        const int padded = (len + 127) & ~127;
#pragma unroll 8
        for (int p = lane; p < padded; p += 32) B[p] = p < len ? bases[o + p] : (uint8_t)'A';
        if (lane < SW) sF[warp][lane] = 0;
        __syncwarp();
        // 4 characters -> 1 byte per lane and 128-base group: code = ((c >> 1) ^ (c >> 2)) & 3 (A0 C1 G2 T3, any case)
        bool invalid = false;
        for (int g = 0; g < padded; g += 128) {
            const u32 x = *reinterpret_cast<const u32 *>(B + g + 4 * lane);
            const u32 up = x & 0xDFDFDFDFu;
            const u32 eqA = up ^ 0x41414141u, eqC = up ^ 0x43434343u, eqG = up ^ 0x47474747u, eqT = up ^ 0x54545454u;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const u32 m = 0xFFu << (8 * t);
                invalid |= (eqA & m) && (eqC & m) && (eqG & m) && (eqT & m);
            }
            const u32 c = ((x >> 1) ^ (x >> 2)) & 0x03030303u;
            const u32 byte = (c * 0x40100401u) >> 24;              // first character in the top two bits
            const int bi = (g >> 2) + lane;                         // byte index in the big-endian 2-bit string
            if (bi < 8 * SW) Fb[(bi & ~7) + 7 - (bi & 7)] = (uint8_t)byte;      // little-endian u64 words in shared memory
        }
        bad |= __any_sync(0xffffffffu, invalid);
        __syncwarp();
        // padding 'A's packed as 0 bits already; reverse complement from the packed words (utils.cpp:73-91)
        if (lane < SW) {
            const int sh = 64 * SW - 2 * len, q = sh >> 6, rr = sh & 63;
            const int i0 = lane + q, i1 = lane + q + 1;
            const u64 a = i0 < SW ? rev2(~sF[warp][SW - 1 - i0]) : 0ull;
            const u64 b2 = i1 < SW ? rev2(~sF[warp][SW - 1 - i1]) : 0ull;
            sR[warp][lane] = rr == 0 ? a : ((a << rr) | (b2 >> (64 - rr)));
        }
        __syncwarp();
        // canonical orientation: keep the read iff read < revcomp (readLoader.cpp:195)
        const u64 f = lane < SW ? sF[warp][lane] : 0ull, qv = lane < SW ? sR[warp][lane] : 0ull;
        const unsigned diff = __ballot_sync(0xffffffffu, f != qv);
        bool use_rc = false;
        if (diff) {
            const int first = __ffs(diff) - 1;
            use_rc = __shfl_sync(0xffffffffu, (int)(qv < f), first) != 0;
        }
        if (lane < SW) {
            u64 v = use_rc ? qv : f;
            if (lane == SW - 1) v |= (u64)len;
            rec[r * SW + lane] = bad ? ~0ull : v;
        }
        if (!bad) { good++; bp += (unsigned long long)len; }
        __syncwarp();
    }
    if (lane == 0 && good) {
        atomicAdd(&counters[0], good);
        atomicAdd(&counters[1], bp);
    }
}

// K1, thread per read.  A block stages the contiguous characters of its reads in shared memory with coalesced
// loads (16 bytes per lane where the alignment allows), then every thread packs, reverse-complements and
// orients ONE read: 32 reads per warp instruction instead of one (the warp-per-read kernel above is issue-bound
// at ~400 instructions per read).  Used when a block's reads fit the staging buffer.
constexpr int K1T_THREADS = 256;
constexpr int K1T_STAGE = 40 * 1024;        // bytes of characters per block

template <int SW>
__global__ void __launch_bounds__(K1T_THREADS) pack_thread_kernel(const uint8_t *__restrict__ bases, const int64_t *__restrict__ off, u64 n, int k,
                                                                    int rpb, u64 *__restrict__ rec, unsigned long long *counters)
{
    __shared__ __align__(16) uint8_t sB[K1T_STAGE + 32];
    __shared__ unsigned long long sCnt[2];
    if (threadIdx.x < 2) sCnt[threadIdx.x] = 0;
    const u64 nblocks = (n + rpb - 1) / rpb;
    unsigned long long good = 0, bp = 0;
    for (u64 blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
        const u64 r0 = blk * (u64)rpb;
        const int nr = (int)((n - r0) < (u64)rpb ? (n - r0) : (u64)rpb);
        const int64_t start = off[r0], end = off[r0 + nr];
        const int64_t a0 = start & ~(int64_t)15;                   // staging keeps the 16-byte phase of the global address
        const int head = (int)(start - a0);
        const int64_t span = end - start;
        __syncthreads();                                           // previous batch fully consumed
        if (span <= K1T_STAGE) {
            const bool aligned = (((uintptr_t)bases) & 15) == 0;
            const int64_t lo16 = (start + 15) & ~(int64_t)15, hi16 = end & ~(int64_t)15;
            if (aligned && hi16 > lo16) {
                for (int64_t g = lo16 + 16 * (int64_t)threadIdx.x; g < hi16; g += 16 * K1T_THREADS)
                    *reinterpret_cast<uint4 *>(sB + (g - a0)) = __ldg(reinterpret_cast<const uint4 *>(bases + g));
                for (int64_t g = start + threadIdx.x; g < lo16; g += K1T_THREADS) sB[g - a0] = bases[g];
                for (int64_t g = hi16 + threadIdx.x; g < end; g += K1T_THREADS) sB[g - a0] = bases[g];
            } else {
                for (int64_t g = start + threadIdx.x; g < end; g += K1T_THREADS) sB[g - a0] = bases[g];
            }
        }
        __syncthreads();
        if ((int)threadIdx.x < nr) {
            const u64 r = r0 + threadIdx.x;
            const int64_t o = off[r];
            const int64_t len64 = off[r + 1] - o;
            const int max_ok = 32 * SW - 8;
            bool bad = len64 <= (int64_t)k || len64 > (int64_t)max_ok;
            const int len = bad ? 0 : (int)len64;
            // (a block whose span does not fit -- only possible next to over-long, rejected reads -- reads global memory)
            const uint8_t *B = span <= K1T_STAGE ? sB + head + (o - start) : bases + o;
            u64 f[SW], q[SW];
#pragma unroll
            for (int w = 0; w < SW; ++w) f[w] = 0;
            bool invalid = false;
            if (span <= K1T_STAGE) {
                // four characters per step out of the staging buffer: two aligned 32-bit words funnel-shifted to the read's
                // byte phase; codes of the four bytes at once ((c >> 1) ^ (c >> 2)) & 3; validity by rebuilding the
                // upper-case character each code stands for (A 0x41, C +2, G +6, T +0x13) and comparing; the four 2-bit
                // codes gathered into one byte by a multiply
                const u32 *Bw = reinterpret_cast<const u32 *>(reinterpret_cast<uintptr_t>(B) & ~(uintptr_t)3);
                const unsigned ph = (unsigned)(reinterpret_cast<uintptr_t>(B) & 3) * 8;
                u32 lo = Bw[0], bad_bits = 0;
#pragma unroll
                for (int w = 0; w < SW; ++w) {
                    u64 acc = 0;
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const int c4 = 8 * w + q;
                        if (4 * c4 < len) {
                            const u32 hi = Bw[c4 + 1];
                            u32 x = __funnelshift_r(lo, hi, ph);
                            lo = hi;
                            const int left = len - 4 * c4;
                            if (left < 4) { const u32 keep = 0xFFFFFFFFu >> (8 * (4 - left)); x = (x & keep) | (0x41414141u & ~keep); }
                            const u32 c = ((x >> 1) ^ (x >> 2)) & 0x03030303u;
                            const u32 c0 = c & 0x01010101u, c1 = (c >> 1) & 0x01010101u;
                            const u32 expect = 0x41414141u + (c0 & ~c1) * 2u + (c1 & ~c0) * 6u + (c1 & c0) * 0x13u;
                            bad_bits |= expect ^ (x & 0xDFDFDFDFu);
                            u32 byte = (c * 0x40100401u) >> 24;
                            if (left < 4) byte &= 0xFFu << (2 * (4 - left));      // padding characters are not bases
                            acc |= (u64)byte << (56 - 8 * q);
                        }
                    }
                    f[w] = acc;
                }
                invalid = bad_bits != 0;
            } else {
#pragma unroll
                for (int w = 0; w < SW; ++w) {
                    if (32 * w < len) {
                        u64 acc = 0;
                        const int m = len - 32 * w < 32 ? len - 32 * w : 32;
                        for (int t = 0; t < m; ++t) {
                            const u32 ch = B[32 * w + t];
                            const u32 up = ch & 0xDFu;
                            invalid |= !(up == 'A' || up == 'C' || up == 'G' || up == 'T');
                            acc |= (u64)(((ch >> 1) ^ (ch >> 2)) & 3u) << (62 - 2 * t);
                        }
                        f[w] = acc;
                    }
                }
            }
            bad |= invalid;
            revcomp_record(f, q, SW, len);          // q[SW-1] carries the length, f does not yet
            f[SW - 1] |= (u64)len;
            bool use_rc = false;                    // keep the read iff read < revcomp (readLoader.cpp:195)
#pragma unroll
            for (int w = SW - 1; w >= 0; --w) if (f[w] != q[w]) use_rc = q[w] < f[w];
#pragma unroll
            for (int w = 0; w < SW; ++w) rec[r * SW + w] = bad ? ~0ull : (use_rc ? q[w] : f[w]);
            if (!bad) { good++; bp += (unsigned long long)len; }
        }
    }
    if (good) { atomicAdd(&sCnt[0], good); atomicAdd(&sCnt[1], bp); }
    __syncthreads();
    if (threadIdx.x == 0 && sCnt[0]) { atomicAdd(&counters[0], sCnt[0]); atomicAdd(&counters[1], sCnt[1]); }
}

// One chunk of the streamed upload: append the bases, append the offsets rebased to the running total.
__global__ void __launch_bounds__(256) rebase_offsets_kernel(const int64_t *__restrict__ in, int64_t n, int64_t delta, int64_t *__restrict__ out)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = in[i] + delta;
}

template <typename T>
static void grow(DevBuf<T> &b, size_t used, size_t need, cudaStream_t st)
{
    if (need <= b.n) return;
    size_t cap = b.n ? b.n : (size_t)1 << 20;
    while (cap < need) cap += cap / 2 + 1;
    DevBuf<T> nb;
    nb.persistent = true;       // moved into a context member below
    nb.alloc(cap, st);
    if (used) SG_CUDA(cudaMemcpyAsync(nb.p, b.p, used * sizeof(T), cudaMemcpyDeviceToDevice, st));
    b = std::move(nb);
}

void stage_upload_chunk(Context &c, const uint8_t *bases, const int64_t *offsets, int64_t n_reads)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    const int64_t first = offsets[0], nb = offsets[n_reads] - first;
    SG_CHECK(nb >= 0, "offsets must be non-decreasing");
    SG_CHECK(c.up_reads + (u64)n_reads < 0x3FFFFFFFull, "at most 2^30-1 reads per context");
    grow(c.up_d_bases, (size_t)c.up_bases, (size_t)(c.up_bases + (u64)nb), st);
    grow(c.up_d_offsets, (size_t)(c.up_reads ? c.up_reads + 1 : 0), (size_t)(c.up_reads + (u64)n_reads + 1), st);
    if (nb) SG_CUDA(cudaMemcpyAsync(c.up_d_bases.p + c.up_bases, bases + first, (size_t)nb, cudaMemcpyHostToDevice, st));
    DevBuf<int64_t> tmp((size_t)n_reads + 1, st);
    SG_CUDA(cudaMemcpyAsync(tmp.p, offsets, ((size_t)n_reads + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    rebase_offsets_kernel<<<grid_for((u64)n_reads + 1, 256, 4), 256, 0, st>>>(tmp.p, n_reads + 1, (int64_t)c.up_bases - first, c.up_d_offsets.p + c.up_reads);
    SG_LAUNCHED();
    c.up_reads += (u64)n_reads;
    c.up_bases += (u64)nb;
}

// longest of the n reads whose (device) offsets are d_o (caller holds an ArenaScope)
static int longest_read(const int64_t *d_o, u64 n, cudaStream_t st)
{
    DevBuf<int> d_max(1, st);
    SG_CUDA(cudaMemsetAsync(d_max.p, 0, sizeof(int), st));
    unsigned g = grid_for(n, K1_WARPS * 32, 4);
    if (g > kSMs * 8) g = kSMs * 8;
    if (n > 0) { max_len_kernel<<<g, K1_WARPS * 32, 0, st>>>(d_o, n, d_max.p); SG_LAUNCHED(); }
    int max_len = 0;
    SG_CUDA(cudaMemcpyAsync(&max_len, d_max.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    return max_len;
}

int stage_uploaded_max_len(Context &c)
{
    ArenaScope arena_scope(c.arena, c.stream);
    return longest_read(c.up_d_offsets.p, c.up_reads, c.stream);
}

void stage_ingest_ascii(Context &c, const uint8_t *bases, const int64_t *offsets, int64_t n_reads, bool device_resident, int forced_max_len)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    SG_CHECK(n_reads >= 0, "negative read count");
    SG_CHECK((u64)n_reads < 0x3FFFFFFFull, "at most 2^30-1 reads per context");
    c.n_input = (u64)n_reads;
    c.have_reads = c.have_table = c.have_graph = false;
    c.cnt = Counters();
    c.cnt.total_reads = (u64)n_reads;
    c.h = hash_len_for(c.min_overlap);
    c.cnt.hash_len = (u64)c.h;
    if (n_reads == 0 && forced_max_len <= 0) { c.SW = 1; c.max_len = 0; c.raw_slice.alloc(0, st); return; }

    const uint8_t *d_b = bases;
    const int64_t *d_o = offsets;
    if (!device_resident) {
        const int64_t total = offsets[n_reads];
        // grow-only staging buffers, kept between calls: re-allocating ~0.5 GB per call made the stream-ordered
        // pool map fresh memory every few calls (hundreds of ms)
        c.d_offsets.alloc((size_t)n_reads + 1, st);
        c.d_bases.alloc((size_t)total, st);
        SG_CUDA(cudaMemcpyAsync(c.d_offsets.p, offsets, ((size_t)n_reads + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        if (total) SG_CUDA(cudaMemcpyAsync(c.d_bases.p, bases, (size_t)total, cudaMemcpyHostToDevice, st));
        d_b = c.d_bases.p; d_o = c.d_offsets.p;
    }
    // longest read decides the record stride
    int max_len = longest_read(d_o, (u64)n_reads, st);
    // The reference has no length limit; this build packs reads of up to 1016 bases (kMaxWords 64-bit words per record).
    // Dropping a longer read silently would renumber every read after it, so the call fails instead.
    SG_CHECK(max_len <= 32 * kMaxWords - 8, "a read is longer than 1016 bases: not supported by this build of libsage2gpu");
    if (forced_max_len > 0) {       // a slice of a read set that several GPUs pack: the record stride follows the longest read of ALL slices
        SG_CHECK(max_len <= forced_max_len, "a read of this slice is longer than the maximum given for the whole read set");
        max_len = forced_max_len;
    }
    if (max_len < 1) max_len = 1;
    c.max_len = max_len;
    c.SW = words_for_len(max_len);
    {   // the search kernels are instantiated for these strides (search.cu SG_DISPATCH_SW)
        static const int kStrides[] = { 2, 3, 4, 5, 6, 8, 12, 16, 32 };
        for (int s : kStrides) if (s >= c.SW) { c.SW = s; break; }
    }

    // K1 (a slice of a partitioned ingest is packed into a buffer of its own: the joint array is c.raw)
    DevBuf<u64> &rec = forced_max_len != 0 ? c.raw_slice : c.raw;       // < 0: a slice whose own longest read decides
    rec.alloc((size_t)n_reads * c.SW, st);
    if (n_reads == 0) { c.cnt.good_reads = 0; c.cnt.total_bp = 0; c.cnt.avg_len = 0; return; }
    DevBuf<unsigned long long> d_cnt(2, st);
    SG_CUDA(cudaMemsetAsync(d_cnt.p, 0, 2 * sizeof(unsigned long long), st));
    int rpb = K1T_STAGE / (max_len > 0 ? max_len : 1);           // reads per block of the thread-per-read kernel
    if (rpb > K1T_THREADS) rpb = K1T_THREADS;
    rpb &= ~31;
    static const bool warp_per_read = getenv("SAGE2GPU_PACK_WARP") != nullptr;
    if (rpb >= 32 && c.SW <= 8 && !warp_per_read) {
        unsigned gp = grid_for((u64)n_reads, 1, (unsigned)rpb);
        if (gp > kSMs * 8) gp = kSMs * 8;
        switch (c.SW) {
            case 2: pack_thread_kernel<2><<<gp, K1T_THREADS, 0, st>>>(d_b, d_o, (u64)n_reads, c.min_overlap, rpb, rec.p, d_cnt.p); break;
            case 3: pack_thread_kernel<3><<<gp, K1T_THREADS, 0, st>>>(d_b, d_o, (u64)n_reads, c.min_overlap, rpb, rec.p, d_cnt.p); break;
            case 4: pack_thread_kernel<4><<<gp, K1T_THREADS, 0, st>>>(d_b, d_o, (u64)n_reads, c.min_overlap, rpb, rec.p, d_cnt.p); break;
            case 5: pack_thread_kernel<5><<<gp, K1T_THREADS, 0, st>>>(d_b, d_o, (u64)n_reads, c.min_overlap, rpb, rec.p, d_cnt.p); break;
            case 6: pack_thread_kernel<6><<<gp, K1T_THREADS, 0, st>>>(d_b, d_o, (u64)n_reads, c.min_overlap, rpb, rec.p, d_cnt.p); break;
            default: pack_thread_kernel<8><<<gp, K1T_THREADS, 0, st>>>(d_b, d_o, (u64)n_reads, c.min_overlap, rpb, rec.p, d_cnt.p); break;
        }
    } else {        // long reads: one warp per read
        unsigned gp = grid_for((u64)n_reads, 1, K1_WARPS);
        if (gp > kSMs * 16) gp = kSMs * 16;
        pack_kernel<<<gp, K1_WARPS * 32, 0, st>>>(d_b, d_o, (u64)n_reads, c.min_overlap, c.SW, rec.p, d_cnt.p);
    }
    SG_LAUNCHED();
    unsigned long long h_cnt[2];
    SG_CUDA(cudaMemcpyAsync(h_cnt, d_cnt.p, sizeof(h_cnt), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    c.cnt.good_reads = h_cnt[0];
    c.cnt.total_bp = h_cnt[1];
    c.cnt.avg_len = h_cnt[0] ? h_cnt[1] / h_cnt[0] : 0;        // readLoader.cpp:161 integer division
}

// ------------------------------------------------------------------------------------------------
// K2: sort a permutation of the good reads by record (= Read::operator<), dedupe.  Six stable 8-bit radix
// passes on the leading 16..24 bases + an in-place fix of the short runs of equal prefixes by whole-record
// compares; inputs with very long runs fall back to LSD passes over every word.
// ------------------------------------------------------------------------------------------------
__global__ void iota_kernel(u32 *v, u64 n)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) v[i] = (u32)i;
}

__global__ void gather_word_kernel(const u64 *__restrict__ rec, const u32 *__restrict__ perm, u64 n, int SW, int w, u64 *__restrict__ key)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        key[i] = rec[(u64)perm[i] * SW + w];
}

__device__ __forceinline__ bool rec_differs(const u64 *a, const u64 *b, int SW)
{
    u64 d = 0;
    for (int w = 0; w < SW; ++w) d |= a[w] ^ b[w];
    return d != 0;
}

// F / RC records are written by groups of SWS / 4 lanes, one 256-bit store of four words per lane: the groups of a warp
// cover consecutive unique ids, so a warp's stores are whole contiguous lines (a lane per record stored every word to
// a different line).  The lanes of a group meet in shared memory to form the reverse complement.
constexpr int UW_THREADS = 256;
__device__ __forceinline__ void ld256(const u64 *p, u64 (&v)[4])
{
    asm volatile("ld.global.nc.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v[0]), "=l"(v[1]), "=l"(v[2]), "=l"(v[3]) : "l"(p));
}
__device__ __forceinline__ void st256(u64 *p, const u64 (&v)[4])
{
    asm volatile("st.global.v4.u64 [%0], {%1,%2,%3,%4};" :: "l"(p), "l"(v[0]), "l"(v[1]), "l"(v[2]), "l"(v[3]) : "memory");
}
// lane g of a group holds words 4g .. 4g+3 of its record in f and the whole record is in grp[]: store both strands' words
template <bool WITH_RC>
__device__ __forceinline__ void store_group_words(const u64 *grp, const u64 (&f)[4], int g, int SW, int len, u64 *Fdst, u64 *RCdst)
{
    st256(Fdst + 4 * g, f);
    if (WITH_RC) {
        u64 r[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { const int w = 4 * g + j; r[j] = w < SW ? revcomp_word(grp, SW, len, w) : 0ull; }
        st256(RCdst + 4 * g, r);
    }
}

template <bool WITH_RC>
__global__ void __launch_bounds__(UW_THREADS) unique_write_kernel(const u64 *__restrict__ rec, const u32 *__restrict__ perm, const u32 *__restrict__ flag,
                                                                   const u32 *__restrict__ uidx, u64 n_good, int SW, int SWS,
                                                                   u64 *__restrict__ F, u64 *__restrict__ RC, uint16_t *__restrict__ len, u32 *__restrict__ start)
{
    __shared__ u64 sRec[UW_THREADS * 4];
    const int G = SWS / 4, g = threadIdx.x & (G - 1);
    const u64 per_block = UW_THREADS / G;
    u64 *grp = sRec + 4 * (threadIdx.x - g);
    for (u64 i0 = (u64)blockIdx.x * per_block; i0 < n_good; i0 += (u64)gridDim.x * per_block) {      // uniform trip count per block
        const u64 i = i0 + threadIdx.x / G;
        const bool active = i < n_good && flag[i];
        u64 f[4] = { 0, 0, 0, 0 };
        if (active) {
            const u64 *a = rec + (u64)perm[i] * SW;
#pragma unroll
            for (int j = 0; j < 4; ++j) { const int w = 4 * g + j; if (w < SW) f[j] = a[w]; grp[4 * g + j] = f[j]; }
        }
        __syncwarp();
        if (active) {
            const u32 u = uidx[i];
            const int l = rec_len(grp, SW);
            store_group_words<WITH_RC>(grp, f, g, SW, l, F + (u64)u * SWS, WITH_RC ? RC + (u64)u * SWS : nullptr);
            if (g == 0) { len[u] = (uint16_t)l; start[u] = (u32)i; }
        }
        __syncwarp();
    }
}

__global__ void freq_kernel(const u32 *__restrict__ start, u64 U, u64 n_good, uint16_t *__restrict__ freq)
{
    for (u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x; u < U; u += (u64)gridDim.x * blockDim.x) {
        const u64 e = (u + 1 < U) ? start[u + 1] : n_good;
        freq[u] = (uint16_t)(e - start[u]);       // uint16_t frequency wraps like readLoader.cpp:234
    }
}

static unsigned big_grid(u64 n, unsigned block = 256)
{
    unsigned g = grid_for(n, block, 4);
    return g > kSMs * 16u ? kSMs * 16u : g;
}

// good reads only: bad ones were packed as all-ones records
__global__ void flag_good_kernel(const u64 *__restrict__ rec, u64 n, int SW, u32 *__restrict__ flag)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        flag[i] = (rec[i * SW + SW - 1] & 0xFFFFull) != 0xFFFFull;
}

__global__ void compact_good_kernel(const u64 *__restrict__ rec, const u32 *__restrict__ flag, const u32 *__restrict__ idx, u64 n, int SW,
                                    u64 *__restrict__ key, u32 *__restrict__ val)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        if (flag[i]) { key[idx[i]] = rec[i * SW]; val[idx[i]] = (u32)i; }
}

// After the sort by the leading bases: order every run of equal prefixes by the whole records, and flag the first read
// of every distinct record (the dedupe).  A read whose prefix differs from its predecessor's is new without a look at
// the records; only the members of runs are compared.
// Runs are short (duplicate reads, shared 24-mers); a run longer than kTieLimit (an insertion sort by one thread would
// be the tail of the kernel) raises `overflow` and is left to refine_long_runs, which flags its members too.
constexpr int kTieLimit = 32;
// The radix passes cover the top 64 - skip bits of the first word: enough bits that runs of equal prefixes stay short
// for the number of reads at hand (n reads spread over 2^(64-skip) prefixes), in whole 8-bit passes: 32 bits (16 bases,
// 4 passes) up to 134 M reads, 40 bits up to 2^35, never more than 48.
static int sort_skip_bits(u64 n)
{
    int lg = 0;
    while (lg < 63 && (1ull << lg) < n) ++lg;
    int bits = ((lg + 5 + 7) / 8) * 8;
    if (bits < 32) bits = 32;
    if (bits > 48) bits = 48;
    return 64 - bits;
}
__device__ __forceinline__ bool rec_less(const u64 *a, const u64 *b, int SW)
{
    for (int w = 0; w < SW; ++w) { const u64 x = a[w], y = b[w]; if (x != y) return x < y; }
    return false;
}
__global__ void __launch_bounds__(256) tie_fix_kernel(const u64 *__restrict__ rec, const u64 *__restrict__ key, u32 *__restrict__ perm, u64 n, int SW,
                                                        int kSortSkipBits, u32 *__restrict__ flag, u32 *__restrict__ overflow)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const u64 k = key[i] >> kSortSkipBits;
        if (i > 0 && (key[i - 1] >> kSortSkipBits) == k) continue;      // a member: its run's head flags it
        flag[i] = 1u;
        if (i + 1 >= n || (key[i + 1] >> kSortSkipBits) != k) continue;      // not the head of a run of >= 2
        u64 e = i + 2;
        while (e < n && (key[e] >> kSortSkipBits) == k && e - i <= (u64)kTieLimit) ++e;
        if (e - i > (u64)kTieLimit) { *overflow = 1u; continue; }
        for (u64 a = i + 1; a < e; ++a) {
            const u32 x = perm[a];
            const u64 *rx = rec + (u64)x * SW;
            u64 b = a;
            while (b > i && rec_less(rx, rec + (u64)perm[b - 1] * SW, SW)) { perm[b] = perm[b - 1]; --b; }
            perm[b] = x;
        }
        for (u64 a = i + 1; a < e; ++a) flag[a] = rec_differs(rec + (u64)perm[a] * SW, rec + (u64)perm[a - 1] * SW, SW) ? 1u : 0u;
    }
}

// ---- runs longer than kTieLimit (reads inside high-copy repeats, low-complexity sequence) ---------------------------
// Only their members are sorted again, by (run, rest of the record): LSD radix passes over a compacted copy, written
// back to the positions the run occupies.  Everything else keeps the order the first-word sort + tie_fix gave it.
__global__ void __launch_bounds__(256) run_boundary_kernel(const u64 *__restrict__ key, u64 n, int kSortSkipBits, u32 *__restrict__ flag)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        flag[i] = (i == 0 || (key[i] >> kSortSkipBits) != (key[i - 1] >> kSortSkipBits)) ? 1u : 0u;
}
__global__ void __launch_bounds__(256) run_count_kernel(const u32 *__restrict__ flag, const u32 *__restrict__ excl, u64 n, u32 *__restrict__ cnt)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        atomicAdd(&cnt[excl[i] + flag[i] - 1], 1u);
}
__global__ void __launch_bounds__(256) run_long_flag_kernel(const u32 *__restrict__ flag, const u32 *__restrict__ excl, const u32 *__restrict__ cnt, u64 n,
                                                            u32 *__restrict__ lflag)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        lflag[i] = cnt[excl[i] + flag[i] - 1] > (u32)kTieLimit ? 1u : 0u;
}
__global__ void __launch_bounds__(256) run_compact_kernel(const u32 *__restrict__ lflag, const u32 *__restrict__ lidx, const u32 *__restrict__ flag,
                                                          const u32 *__restrict__ excl, const u32 *__restrict__ perm, u64 n,
                                                          u32 *__restrict__ pos, u32 *__restrict__ val, u64 *__restrict__ run)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        if (lflag[i]) { const u32 j = lidx[i]; pos[j] = (u32)i; val[j] = perm[i]; run[j] = (u64)(excl[i] + flag[i] - 1); }
}
__global__ void __launch_bounds__(256) run_scatter_kernel(const u32 *__restrict__ pos, const u32 *__restrict__ val, u64 m, u32 *__restrict__ perm)
{
    for (u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x; j < m; j += (u64)gridDim.x * blockDim.x) perm[pos[j]] = val[j];
}
// after the scatter: the dedupe flag of the members (a run's head is flagged by tie_fix_kernel already)
__global__ void __launch_bounds__(256) run_member_flag_kernel(const u64 *__restrict__ rec, const u32 *__restrict__ pos, const u32 *__restrict__ bound,
                                                              const u32 *__restrict__ perm, u64 m, int SW, u32 *__restrict__ flag)
{
    for (u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x; j < m; j += (u64)gridDim.x * blockDim.x) {
        const u32 i = pos[j];
        if (!bound[i]) flag[i] = rec_differs(rec + (u64)perm[i] * SW, rec + (u64)perm[i - 1] * SW, SW) ? 1u : 0u;
    }
}

// returns m, the members of the runs longer than kTieLimit
static u32 refine_long_runs(Context &c, const u64 *rec, const u64 *key, u32 *perm, u64 n, int SW, int kSortSkipBits, u32 *dedupe_flag)
{
    cudaStream_t st = c.stream;
    DevBuf<u32> bound(n, st), excl(n, st), cnt(n, st), lflag(n, st), lidx(n, st), d_m(1, st);
    run_boundary_kernel<<<big_grid(n), 256, 0, st>>>(key, n, kSortSkipBits, bound.p);
    SG_LAUNCHED();
    exclusive_scan_u32(bound.p, excl.p, n, nullptr, st);
    SG_CUDA(cudaMemsetAsync(cnt.p, 0, n * sizeof(u32), st));
    run_count_kernel<<<big_grid(n), 256, 0, st>>>(bound.p, excl.p, n, cnt.p);
    SG_LAUNCHED();
    run_long_flag_kernel<<<big_grid(n), 256, 0, st>>>(bound.p, excl.p, cnt.p, n, lflag.p);
    SG_LAUNCHED();
    exclusive_scan_u32(lflag.p, lidx.p, n, d_m.p, st);
    u32 m = 0;
    SG_CUDA(cudaMemcpyAsync(&m, d_m.p, sizeof(u32), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    if (m == 0) return 0;
    DevBuf<u32> pos(m, st), v0(m, st), v1(m, st);
    DevBuf<u64> a0(m, st), a1(m, st), b0(m, st), b1(m, st);
    run_compact_kernel<<<big_grid(n), 256, 0, st>>>(lflag.p, lidx.p, bound.p, excl.p, perm, n, pos.p, v0.p, b0.p);
    SG_LAUNCHED();
    SortCols cols;
    cols.a[0] = a0.p; cols.a[1] = a1.p; cols.b[0] = b0.p; cols.b[1] = b1.p; cols.v[0] = v0.p; cols.v[1] = v1.p;
    int cur = 0;
    for (int w = SW - 1; w >= 0; --w) {      // least significant word first; of the first word only the bits the first sort skipped
        gather_word_kernel<<<big_grid(m), 256, 0, st>>>(rec, cols.v[cur], m, SW, w, cols.a[cur]);
        SG_LAUNCHED();
        cur = radix_sort_bits(cols, cur, m, false, 0, w == 0 ? kSortSkipBits : 64, st);
    }
    int id_bits = 1;
    while ((n >> id_bits) != 0) ++id_bits;
    cur = radix_sort_bits(cols, cur, m, true, 0, id_bits, st);      // ... and the run last: members return to their run's positions
    run_scatter_kernel<<<big_grid(m), 256, 0, st>>>(pos.p, cols.v[cur], m, perm);
    SG_LAUNCHED();
    run_member_flag_kernel<<<big_grid(m), 256, 0, st>>>(rec, pos.p, bound.p, perm, m, SW, dedupe_flag);
    SG_LAUNCHED();
    return m;
}

// ---- several GPUs: rank r organises the reads whose leading bases fall into its key range ------------------------
// Every rank holds all packed records (the input is replicated or all-gathered), so the splitters -- quantiles of a
// 4096-bin histogram of the leading 6 bases -- come out identical everywhere without an exchange; equal records share
// a bin, so the dedupe stays local and the ranks' unique runs concatenate to the global sorted order.
constexpr int kSplitBits = 12;
__global__ void __launch_bounds__(256) split_hist_kernel(const u64 *__restrict__ key, u64 n, u32 *__restrict__ hist)
{
    __shared__ u32 sh[1 << kSplitBits];
    for (int b = threadIdx.x; b < (1 << kSplitBits); b += blockDim.x) sh[b] = 0;
    __syncthreads();
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) atomicAdd(&sh[key[i] >> (64 - kSplitBits)], 1u);
    __syncthreads();
    for (int b = threadIdx.x; b < (1 << kSplitBits); b += blockDim.x) if (sh[b]) atomicAdd(&hist[b], sh[b]);
}
__global__ void __launch_bounds__(256) split_flag_kernel(const u64 *__restrict__ key, u64 n, u32 lo_bin, u32 hi_bin, u32 *__restrict__ flag)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const u32 b = (u32)(key[i] >> (64 - kSplitBits));
        flag[i] = (b >= lo_bin && b < hi_bin) ? 1u : 0u;
    }
}
__global__ void __launch_bounds__(256) split_compact_kernel(const u64 *__restrict__ key, const u32 *__restrict__ val, const u32 *__restrict__ flag,
                                                            const u32 *__restrict__ idx, u64 n, u64 *__restrict__ okey, u32 *__restrict__ oval)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        if (flag[i]) { okey[idx[i]] = key[i]; oval[idx[i]] = val[i]; }
}
__global__ void __launch_bounds__(UW_THREADS) revcomp_range_kernel(const u64 *__restrict__ F, u64 *__restrict__ RC, const uint16_t *__restrict__ len,
                                                                   u64 U, int SW, int SWS)
{
    __shared__ u64 sRec[UW_THREADS * 4];
    const int G = SWS / 4, g = threadIdx.x & (G - 1);
    const u64 per_block = UW_THREADS / G;
    u64 *grp = sRec + 4 * (threadIdx.x - g);
    for (u64 u0 = (u64)blockIdx.x * per_block; u0 < U; u0 += (u64)gridDim.x * per_block) {
        const u64 u = u0 + threadIdx.x / G;
        u64 f[4] = { 0, 0, 0, 0 };
        if (u < U) {
            ld256(F + u * SWS + 4 * g, f);
#pragma unroll
            for (int j = 0; j < 4; ++j) grp[4 * g + j] = f[j];
        }
        __syncwarp();
        if (u < U) {
            u64 r[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) { const int w = 4 * g + j; r[j] = w < SW ? revcomp_word(grp, SW, (int)len[u], w) : 0ull; }
            st256(RC + u * SWS + 4 * g, r);
        }
        __syncwarp();
    }
}

void stage_organize_reads(Context &c, int rank, int world)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    SG_CHECK(world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world, "bad rank / world");
    const u64 n = c.n_input;
    u64 n_good = c.cnt.good_reads;
    const int SW = c.SW;
    c.cnt.unique_reads = 0;
    c.rp_rank = rank; c.rp_world = world; c.rp_local = 0;
    if (n == 0 || n_good == 0) {
        if (world == 1) { c.F.release(); c.RC.release(); c.len.release(); c.freq.release(); }
        c.have_reads = world == 1;
        return;
    }
    DevBuf<u64> &rec = c.raw;      // packed canonical records in input order (bad reads all-ones)
    DevBuf<u64> ka(n_good, st), kb(n_good, st);
    DevBuf<u32> va(n_good, st), vb(n_good, st);
    {   // indices and first words of the good reads, input order
        DevBuf<u32> gflag(n, st), gidx(n, st);
        flag_good_kernel<<<big_grid(n), 256, 0, st>>>(rec.p, n, SW, gflag.p);
        SG_LAUNCHED();
        exclusive_scan_u32(gflag.p, gidx.p, n, nullptr, st);
        compact_good_kernel<<<big_grid(n), 256, 0, st>>>(rec.p, gflag.p, gidx.p, n, SW, ka.p, va.p);
        SG_LAUNCHED();
    }
    SortCols cols;
    cols.a[0] = ka.p; cols.a[1] = kb.p; cols.b[0] = cols.b[1] = nullptr; cols.v[0] = va.p; cols.v[1] = vb.p;
    const int kSortSkipBits = sort_skip_bits(n_good);       // from the global count: the same passes on every rank
    int cur = 0;
    if (world > 1) {        // keep this rank's key range only
        const int nbins = 1 << kSplitBits;
        DevBuf<u32> hist(nbins, st);
        SG_CUDA(cudaMemsetAsync(hist.p, 0, nbins * sizeof(u32), st));
        split_hist_kernel<<<kSMs * 4, 256, 0, st>>>(ka.p, n_good, hist.p);
        SG_LAUNCHED();
        std::vector<u32> h(nbins);
        SG_CUDA(cudaMemcpyAsync(h.data(), hist.p, nbins * sizeof(u32), cudaMemcpyDeviceToHost, st));
        SG_CUDA(cudaStreamSynchronize(st));
        // bin boundaries: rank r takes bins [bound[r], bound[r+1]); bound[r] = first bin whose prefix reaches r * n_good / world
        std::vector<u32> bound(world + 1, (u32)nbins);
        bound[0] = 0;
        u64 pre = 0;
        int r = 1;
        for (int b = 0; b < nbins && r < world; ++b) {
            while (r < world && pre >= (n_good * (u64)r + (u64)world - 1) / (u64)world) bound[r++] = (u32)b;
            pre += h[b];
        }
        u64 n_part = 0;
        for (u32 b = bound[rank]; b < bound[rank + 1]; ++b) n_part += h[b];
        DevBuf<u32> sflag(n_good, st), sidx(n_good, st);
        split_flag_kernel<<<big_grid(n_good), 256, 0, st>>>(ka.p, n_good, bound[rank], bound[rank + 1], sflag.p);
        SG_LAUNCHED();
        exclusive_scan_u32(sflag.p, sidx.p, n_good, nullptr, st);
        split_compact_kernel<<<big_grid(n_good), 256, 0, st>>>(ka.p, va.p, sflag.p, sidx.p, n_good, kb.p, vb.p);
        SG_LAUNCHED();
        cur = 1;
        n_good = n_part;
        if (n_good == 0) return;
    }
    cur = radix_sort_bits(cols, cur, n_good, false, kSortSkipBits, 64, st);      // 4 .. 6 passes on the leading bases
    // dedupe flags: tie_fix_kernel writes all of them but those of the members of runs longer than kTieLimit, which
    // refine_long_runs sorts again by the rest of the record and flags (high-copy repeats, low-complexity input)
    DevBuf<u32> d_flags(2, st);          // [0] tie-run overflow, [1] unique count
    SG_CUDA(cudaMemsetAsync(d_flags.p, 0, 2 * sizeof(u32), st));
    DevBuf<u32> flag(n_good, st), uidx(n_good, st);
    tie_fix_kernel<<<big_grid(n_good), 256, 0, st>>>(rec.p, cols.a[cur], cols.v[cur], n_good, SW, kSortSkipBits, flag.p, d_flags.p);
    SG_LAUNCHED();
    u32 h_flags[2] = { 0, 0 };
    SG_CUDA(cudaMemcpyAsync(h_flags, d_flags.p, sizeof(u32), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    u32 m_long = 0;
    if (h_flags[0]) m_long = refine_long_runs(c, rec.p, cols.a[cur], cols.v[cur], n_good, SW, kSortSkipBits, flag.p);
    exclusive_scan_u32(flag.p, uidx.p, n_good, d_flags.p + 1, st);
    SG_CUDA(cudaMemcpyAsync(h_flags + 1, d_flags.p + 1, sizeof(u32), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    if (stage_stats_enabled())
        fprintf(stderr, "sage2gpu stats: organize_reads reads=%llu long_run_members=%u unique=%u\n", (unsigned long long)n_good, m_long, h_flags[1]);
    const u32 *perm = cols.v[cur];
    const u32 U = h_flags[1];
    c.cnt.unique_reads = U;
    c.SWS = storage_words(SW);
    // several GPUs: the run goes to buffers of its own and moves into the global arrays once the ranks' counts are known
    // (all of them grow-only: no multi-GB allocation per call)
    DevBuf<u64> &Fo = world > 1 ? c.F_loc : c.F;
    DevBuf<uint16_t> &lo = world > 1 ? c.len_loc : c.len, &fo = world > 1 ? c.freq_loc : c.freq;
    Fo.alloc((size_t)U * c.SWS, st);
    lo.alloc(U, st);
    fo.alloc(U, st);
    DevBuf<u32> start(U, st);
    const unsigned uw_grid = big_grid(n_good * (c.SWS / 4), UW_THREADS);
    if (world > 1) {
        unique_write_kernel<false><<<uw_grid, UW_THREADS, 0, st>>>(rec.p, perm, flag.p, uidx.p, n_good, SW, c.SWS, Fo.p, nullptr, lo.p, start.p);
    } else {
        c.RC.alloc((size_t)U * c.SWS, st);
        unique_write_kernel<true><<<uw_grid, UW_THREADS, 0, st>>>(rec.p, perm, flag.p, uidx.p, n_good, SW, c.SWS, Fo.p, c.RC.p, lo.p, start.p);
    }
    SG_LAUNCHED();
    freq_kernel<<<big_grid(U), 256, 0, st>>>(start.p, U, n_good, fo.p);
    SG_LAUNCHED();
    c.rp_local = U;
    c.have_reads = world == 1;      // several GPUs: complete only after the ranks' runs were gathered (stage_reads_gather_*)
    if (c.opt_low_memory) { SG_CUDA(cudaStreamSynchronize(st)); c.raw.release(); trim_default_pool(c.device, st); }      // the packed input is not needed again
}

// The ranks' unique runs -> the global arrays.  counts[q] = unique reads of rank q (the host all-gathered them): this rank's
// run moves to its place in arrays of the total size, whose device pointers go back to the host for the all-gather.
void stage_reads_gather_layout(Context &c, const u64 *counts, void **F, void **len, void **freq, u64 *first, u64 *total)
{
    cudaStream_t st = c.stream;
    SG_CHECK(c.rp_world > 1 && counts != nullptr, "sage2gpu_load_reads_partition must run first");
    SG_CHECK(counts[c.rp_rank] == c.rp_local, "this rank's count does not match its organised reads");
    u64 tot = 0, base = 0;
    for (int q = 0; q < c.rp_world; ++q) { if (q < c.rp_rank) base += counts[q]; tot += counts[q]; }
    SG_CHECK(tot < 0x3FFFFFFFull, "at most 2^30-1 unique reads");
    c.SWS = storage_words(c.SW);
    c.F.alloc((size_t)tot * c.SWS, st); c.RC.alloc((size_t)tot * c.SWS, st); c.len.alloc(tot, st); c.freq.alloc(tot, st);
    if (c.rp_local) {
        SG_CUDA(cudaMemcpyAsync(c.F.p + base * c.SWS, c.F_loc.p, (size_t)c.rp_local * c.SWS * sizeof(u64), cudaMemcpyDeviceToDevice, st));
        SG_CUDA(cudaMemcpyAsync(c.len.p + base, c.len_loc.p, (size_t)c.rp_local * sizeof(uint16_t), cudaMemcpyDeviceToDevice, st));
        SG_CUDA(cudaMemcpyAsync(c.freq.p + base, c.freq_loc.p, (size_t)c.rp_local * sizeof(uint16_t), cudaMemcpyDeviceToDevice, st));
    }
    SG_CUDA(cudaStreamSynchronize(st));
    c.rp_first = base; c.rp_total = tot;
    if (F) *F = c.F.p;
    if (len) *len = c.len.p;
    if (freq) *freq = c.freq.p;
    if (first) *first = base;
    if (total) *total = tot;
}

// after the all-gather: reverse complements of all reads (utils.cpp:73-91 on packed words), the reads are complete
void stage_reads_gather_finish(Context &c)
{
    cudaStream_t st = c.stream;
    SG_CHECK(c.rp_world > 1, "sage2gpu_load_reads_partition must run first");
    const u64 U = c.rp_total;
    if (U) {
        revcomp_range_kernel<<<big_grid(U * (c.SWS / 4), UW_THREADS), UW_THREADS, 0, st>>>(c.F.p, c.RC.p, c.len.p, U, c.SW, c.SWS);
        SG_LAUNCHED();
    }
    c.cnt.unique_reads = U;
    c.have_reads = true;
    if (c.opt_low_memory) { SG_CUDA(cudaStreamSynchronize(st)); c.F_loc.release(); c.len_loc.release(); c.freq_loc.release(); }
}

// ---- several GPUs, partitioned ingest: every rank packs its slice of the input, the packed records are all-gathered ----
// layout: room for the records of all slices back to back (counts[q] reads of rank q), this rank's slice in place
void stage_raw_gather_layout(Context &c, int rank, int world, const u64 *counts, void **raw, u64 *first, u64 *total)
{
    cudaStream_t st = c.stream;
    SG_CHECK(world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world && counts, "bad rank / world");
    SG_CHECK(counts[rank] == c.n_input, "this rank's count does not match its packed slice");
    u64 tot = 0, base = 0;
    for (int q = 0; q < world; ++q) { if (q < rank) base += counts[q]; tot += counts[q]; }
    SG_CHECK(tot < 0x3FFFFFFFull, "at most 2^30-1 reads");
    c.raw.alloc((size_t)tot * c.SW, st);
    if (c.n_input) SG_CUDA(cudaMemcpyAsync(c.raw.p + base * c.SW, c.raw_slice.p, (size_t)c.n_input * c.SW * sizeof(u64), cudaMemcpyDeviceToDevice, st));
    SG_CUDA(cudaStreamSynchronize(st));
    if (raw) *raw = c.raw.p;
    if (first) *first = base;
    if (total) *total = tot;
    c.rg_total = tot;
}

// after the all-gather: the context holds the packed records of the whole input; the counters are the sums over the slices
void stage_raw_gather_finish(Context &c, u64 total_reads, u64 good_reads, u64 total_bp)
{
    SG_CHECK(c.rg_total == total_reads, "sage2gpu_raw_gather_layout must run first");
    c.n_input = total_reads;
    c.cnt.total_reads = total_reads;
    c.cnt.good_reads = good_reads;
    c.cnt.total_bp = total_bp;
    c.cnt.avg_len = good_reads ? total_bp / good_reads : 0;        // readLoader.cpp:161 integer division
    if (c.opt_low_memory) { SG_CUDA(cudaStreamSynchronize(c.stream)); c.raw_slice.release(); }
}

// ---- a saved .reads file (parse.cu): its lines are the unique reads already, in id order -------------------------------
// Packed by K1 at the stride of the longest read of all slices, then written by the F / RC writer of organizeReads with the
// identity as the sorted order and every read flagged new; the frequencies are the file's.
void stage_pack_saved_reads(Context &c, int rank, int world, int max_len)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    SG_CHECK(world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world, "bad rank / world");
    SG_CHECK(world == 1 || max_len >= 1, "the longest read of the whole read set must be given");
    const u64 n = c.up_reads;
    // the parse already applied isGoodRead's rules (longer than k, ACGT only, at most 1016 bases) and canonical orientation,
    // so K1 drops nothing and keeps F as it is
    stage_ingest_ascii(c, c.up_d_bases.p, c.up_d_offsets.p, (int64_t)n, true, world == 1 && n == 0 ? 0 : max_len);
    SG_CHECK(c.cnt.good_reads == n, "a parsed line was dropped by the pack");
    c.up_d_bases.release(); c.up_d_offsets.release();
    c.rp_rank = rank; c.rp_world = world; c.rp_local = n;
    c.cnt.unique_reads = world == 1 ? n : 0;
    c.SWS = storage_words(c.SW);
    c.have_reads = false;
    if (n == 0) {
        if (world == 1) { c.F.release(); c.RC.release(); c.len.release(); c.freq.release(); }
        c.up_d_freq.release();
        return;
    }
    DevBuf<u64> &Fo = world > 1 ? c.F_loc : c.F;
    DevBuf<uint16_t> &lo = world > 1 ? c.len_loc : c.len, &fo = world > 1 ? c.freq_loc : c.freq;
    Fo.alloc((size_t)n * c.SWS, st);
    lo.alloc(n, st);
    fo.alloc(n, st);
    DevBuf<u32> ids(n, st), ones(n, st), start(n, st);
    iota_kernel<<<big_grid(n), 256, 0, st>>>(ids.p, n);
    SG_LAUNCHED();
    SG_CUDA(cudaMemsetAsync(ones.p, 0x01, n * sizeof(u32), st));
    const unsigned uw_grid = big_grid(n * (c.SWS / 4), UW_THREADS);
    if (world > 1) {
        unique_write_kernel<false><<<uw_grid, UW_THREADS, 0, st>>>(c.raw_slice.p, ids.p, ones.p, ids.p, n, c.SW, c.SWS, Fo.p, nullptr, lo.p, start.p);
    } else {
        c.RC.alloc((size_t)n * c.SWS, st);
        unique_write_kernel<true><<<uw_grid, UW_THREADS, 0, st>>>(c.raw_slice.p, ids.p, ones.p, ids.p, n, c.SW, c.SWS, Fo.p, c.RC.p, lo.p, start.p);
    }
    SG_LAUNCHED();
    SG_CUDA(cudaMemcpyAsync(fo.p, c.up_d_freq.p, n * sizeof(uint16_t), cudaMemcpyDeviceToDevice, st));
    SG_CUDA(cudaStreamSynchronize(st));
    c.up_d_freq.release();
    if (c.opt_low_memory) { c.raw_slice.release(); trim_default_pool(c.device, st); }
}

// first i >= 1 with record i-1 not below record i (Read::operator<: strictly increasing ids, no duplicates)
__global__ void __launch_bounds__(256) order_check_kernel(const u64 *__restrict__ F, u64 U, int SW, int SWS, unsigned long long *first_bad)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x + 1; i < U; i += (u64)gridDim.x * blockDim.x)
        if (!rec_less(F + (i - 1) * SWS, F + i * SWS, SW)) atomicMin(first_bad, (unsigned long long)i);
}

// The complete reads (one context, or after reads_gather_finish): their order, their count against the first line, and the
// counters of step 1 -- good reads = total reads = sum of FREQ, total_bp = sum of FREQ * LEN (readLoader.cpp:161-169)
void stage_check_saved_reads(Context &c, u64 n_reads, u64 good_reads, u64 total_bp)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    SG_CHECK(c.rp_world == 1 || c.have_reads, "sage2gpu_reads_gather_finish must run first");
    const u64 U = c.rp_world == 1 ? c.rp_local : c.cnt.unique_reads;
    c.have_reads = c.have_table = c.have_graph = false;
    if (U > 1) {
        DevBuf<unsigned long long> d_bad(1, st);
        SG_CUDA(cudaMemsetAsync(d_bad.p, 0xFF, sizeof(unsigned long long), st));
        order_check_kernel<<<big_grid(U), 256, 0, st>>>(c.F.p, U, c.SW, c.SWS, d_bad.p);
        SG_LAUNCHED();
        unsigned long long bad = 0;
        SG_CUDA(cudaMemcpyAsync(&bad, d_bad.p, sizeof(bad), cudaMemcpyDeviceToHost, st));
        SG_CUDA(cudaStreamSynchronize(st));
        if (bad != ~0ull)
            throw FormatError(bad + 2, "F is not greater than the F of the line before: the reads must be unique and in increasing order (Read::operator<)");
    }
    if (U < n_reads)
        throw FormatError(U + 2, "the file ends after " + std::to_string(U) + " reads; its first line says " + std::to_string(n_reads));
    if (U > n_reads) throw FormatError(n_reads + 2, "more reads than the " + std::to_string(n_reads) + " its first line says");
    c.cnt.unique_reads = U;
    c.cnt.total_reads = c.cnt.good_reads = good_reads;
    c.cnt.total_bp = total_bp;
    c.cnt.avg_len = good_reads ? total_bp / good_reads : 0;        // readLoader.cpp:161 integer division
    c.h = hash_len_for(c.min_overlap);
    c.cnt.hash_len = (u64)c.h;
    c.have_reads = true;
}

}  // namespace sg
