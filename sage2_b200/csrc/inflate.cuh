// inflate.cuh -- the warp-lockstep DEFLATE decoder (RFC 1951) shared by the BGZF member inflate (inflate.cu) and the range
// decoder of single-member gzip (gunzip.cu).
//
// Every lane of a warp runs the same decoder in lockstep on the same bits -- the loads are broadcasts and the control flow
// stays uniform -- while the lanes share the work that has width: filling the Huffman lookup tables, match copies, stored
// blocks and the CRC32 of the output (per-lane segments combined with the shift operators of zlib's crc32_combine).  Every
// bound is checked before the access it guards.
#pragma once
#include "context.h"

namespace sg {
namespace infl {

constexpr int kLitFast = 10;            // bits of the first-level literal/length table
constexpr int kDistFast = 8;            // bits of the first-level distance table
constexpr u32 kPoly = 0xedb88320u;      // CRC-32 (reflected)
constexpr u32 kWindow = 32768;          // DEFLATE's largest distance
constexpr uint16_t kMarker = 0x8000;    // marker symbol: 0x8000 | position in the 32 KiB window before a range's first byte

// per-warp Huffman state in shared memory: canonical codes as counts per length + symbols in code order (puff's form),
// and first-level tables of (symbol | length << 12) for codes of at most kLitFast / kDistFast bits (0: longer code)
struct Huff {
    uint16_t lfast[1 << kLitFast];
    uint16_t dfast[1 << kDistFast];
    uint16_t lsym[288], dsym[32];
    uint16_t lcount[16], dcount[16];
    uint8_t lens[288 + 32];
};

static __constant__ uint16_t c_lbase[29] = { 3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258 };
static __constant__ uint8_t c_lext[29] = { 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0 };
static __constant__ uint16_t c_dbase[30] = { 1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769,
                                             1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577 };
static __constant__ uint8_t c_dext[30] = { 0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13 };
static __constant__ uint8_t c_clorder[19] = { 16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15 };

// LSB-first bit reader over in[0, end).  Bytes past `end` read as zeros and are never loaded; overrun() says whether the
// bits taken so far reach past `end`.
struct Bits {
    const uint8_t *in;
    u32 end, pos;
    int cnt;
    unsigned long long buf;
    __device__ void refill()
    {
        while (cnt <= 56) {
            const u32 b = pos < end ? in[pos] : 0u;
            ++pos;
            buf |= (unsigned long long)b << cnt;
            cnt += 8;
        }
    }
    __device__ u32 peek(int n) const { return (u32)(buf & ((1ull << n) - 1)); }
    __device__ void drop(int n) { buf >>= n; cnt -= n; }
    __device__ u32 take(int n) { const u32 v = peek(n); drop(n); return v; }
    __device__ unsigned long long taken() const { return 8ull * pos - (unsigned long long)cnt; }
    __device__ bool overrun() const { return taken() > 8ull * end; }
    __device__ void seek(u32 byte) { pos = byte; cnt = 0; buf = 0; }
};

// puff's canonical decode over the next bits of `b` (no bits dropped): the symbol and its length, or -1 (no such code)
__device__ __forceinline__ int slow_decode(const Bits &b, const uint16_t *count, const uint16_t *sym, int &len)
{
    int code = 0, first = 0, index = 0;
    for (int l = 1; l <= 15; ++l) {
        code |= (int)((b.buf >> (l - 1)) & 1u);
        const int n = count[l];
        if (code - n < first) { len = l; return sym[index + (code - first)]; }
        index += n;
        first = (first + n) << 1;
        code <<= 1;
    }
    return -1;
}

__device__ __forceinline__ int decode(Bits &b, const uint16_t *fast, int fast_bits, const uint16_t *count, const uint16_t *sym)
{
    const u32 e = fast[b.peek(fast_bits)];
    if (e) { b.drop((int)(e >> 12)); return (int)(e & 0x1FF); }
    int len = 0;
    const int s = slow_decode(b, count, sym, len);
    if (s >= 0) b.drop(len);
    return s;
}

// puff's `left` of a code with count[l] codes of length l among n symbols: 0 complete (or no codes at all), < 0
// over-subscribed, > 0 incomplete
template <typename C>
__host__ __device__ __forceinline__ int code_left(const C *count, int n)
{
    if ((int)count[0] == n) return 0;
    int left = 1;
    for (int l = 1; l < 16; ++l) {
        left <<= 1;
        left -= (int)count[l];
        if (left < 0) break;
    }
    return left;
}

// a literal/length or distance code the decoder accepts: complete, or a single one-bit code (zlib's inflate_table accepts
// that one)
template <typename C>
__host__ __device__ __forceinline__ bool code_usable(const C *count, int n)
{
    const int left = code_left(count, n);
    return left == 0 || (left > 0 && n == (int)count[0] + (int)count[1]);
}

// count / sym of the code with lengths[0, n) (lane 0), then the first-level table (all lanes).  Returns code_left.
__device__ inline int build_code(const uint8_t *lengths, int n, uint16_t *count, uint16_t *sym, uint16_t *fast, int fast_bits, int lane)
{
    __syncwarp();
    if (lane == 0) {
        uint16_t offs[16];
        for (int l = 0; l < 16; ++l) count[l] = 0;
        for (int s = 0; s < n; ++s) count[lengths[s]]++;
        offs[1] = 0;
        for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + count[l];
        for (int s = 0; s < n; ++s) if (lengths[s]) sym[offs[lengths[s]]++] = (uint16_t)s;
    }
    __syncwarp();
    const int left = code_left(count, n);
    if (fast) {
        for (u32 e = lane; e < (1u << fast_bits); e += 32) {
            int code = 0, first = 0, index = 0;
            uint16_t v = 0;
            for (int l = 1; l <= fast_bits; ++l) {
                code |= (int)((e >> (l - 1)) & 1u);
                const int c = count[l];
                if (code - c < first) { v = (uint16_t)(sym[index + (code - first)] | (l << 12)); break; }
                index += c;
                first = (first + c) << 1;
                code <<= 1;
            }
            fast[e] = v;
        }
    }
    __syncwarp();
    return left;
}

// zlib's multmodp / x2nmodp: products modulo the CRC polynomial, x^(8n)
__host__ __device__ __forceinline__ u32 multmodp(u32 a, u32 b)
{
    u32 m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ kPoly : b >> 1;
    }
    return p;
}

__host__ __device__ __forceinline__ u32 x2nmodp(const u32 *x2n, u64 n, int k)
{
    u32 p = 1u << 31;
    while (n) {
        if (n & 1) p = multmodp(x2n[k & 31], p);
        n >>= 1;
        ++k;
    }
    return p;
}

// the byte-wise CRC table and x^(2^k) of zlib's crc32_combine (block-wide, shared memory)
__device__ inline void crc_tables(u32 *table, u32 *x2n)
{
    for (u32 i = threadIdx.x; i < 256; i += blockDim.x) {
        u32 c = i;
        for (int k = 0; k < 8; ++k) c = c & 1 ? (c >> 1) ^ kPoly : c >> 1;
        table[i] = c;
    }
    if (threadIdx.x == 0) {
        u32 p = 1u << 30;                                  // x^1
        x2n[0] = p;
        for (int k = 1; k < 32; ++k) x2n[k] = p = multmodp(p, p);
    }
    __syncthreads();
}

// CRC32 of out[0, n), the warp's lanes over contiguous segments, combined as crc32_combine does
__device__ inline u32 warp_crc32(const uint8_t *out, u32 n, const u32 *table, const u32 *x2n, int lane)
{
    const u32 seg = (n + 31) / 32, a = min(n, lane * seg), e = min(n, a + seg);
    u32 c = 0xffffffffu;
    for (u32 i = a; i < e; ++i) c = table[(c ^ out[i]) & 0xff] ^ (c >> 8);
    u32 crc = ~c, len = e - a;
    for (int s = 1; s < 32; s <<= 1) {
        const u32 oc = __shfl_down_sync(0xffffffffu, crc, s), ol = __shfl_down_sync(0xffffffffu, len, s);
        if ((lane & (2 * s - 1)) == 0) { crc = multmodp(x2nmodp(x2n, ol, 3), crc) ^ oc; len += ol; }
    }
    return __shfl_sync(0xffffffffu, crc, 0);
}

// One block from its BTYPE on (BFINAL already taken): out[op ..] gets its output and op moves past it.  A distance may reach
// back to out[lo] at most -- the member's first byte -- unless `markers`: then (T = uint16_t, lo = 0, the member began before
// out[0]) a byte before out[0] is written as the marker kMarker | (kWindow + its position), and jmin becomes the lowest
// window position such a marker names.  Returns 0 or a BgzfCode; a caller turns an error met past the end of the data into
// BGZF_TRUNCATED.
template <typename T>
__device__ u32 inflate_block(Bits &b, Huff &h, T *out, u32 &op, u32 out_len, u32 lo, bool markers, u32 &jmin, int lane)
{
    const u32 type = b.take(2);
    if (type == 3) return BGZF_BLOCK_TYPE;
    if (type == 0) {                                   // stored: byte-aligned LEN, NLEN, LEN bytes
        b.drop(b.cnt & 7);
        const u32 len = b.take(16), nlen = b.take(16);
        if (b.overrun()) return BGZF_TRUNCATED;
        if (len != (~nlen & 0xffffu)) return BGZF_STORED_LEN;
        const u32 src = (u32)(b.taken() >> 3);
        if ((u64)src + len > b.end) return BGZF_TRUNCATED;
        if ((u64)op + len > out_len) return BGZF_OUTPUT_OVERFLOW;
        for (u32 t = lane; t < len; t += 32) out[op + t] = (T)b.in[src + t];
        op += len;
        b.seek(src + len);
        __syncwarp();
        return 0;
    }
    if (type == 1) {                                   // fixed codes (RFC 1951 3.2.6)
        if (lane == 0) {
            for (int s = 0; s < 288; ++s) h.lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
            for (int s = 0; s < 30; ++s) h.lens[288 + s] = 5;
        }
        __syncwarp();
        build_code(h.lens, 288, h.lcount, h.lsym, h.lfast, kLitFast, lane);
        build_code(h.lens + 288, 30, h.dcount, h.dsym, h.dfast, kDistFast, lane);
    } else {                                           // dynamic codes (RFC 1951 3.2.7; the checks of puff.c's dynamic())
        const int nlen = (int)b.take(5) + 257, ndist = (int)b.take(5) + 1, ncode = (int)b.take(4) + 4;
        if (nlen > 286 || ndist > 30) return BGZF_BAD_CODE_LENGTHS;
        b.refill();
        __syncwarp();
        if (lane < 19) h.lens[lane] = 0;
        __syncwarp();
        for (int i = 0; i < ncode; ++i) {
            const uint8_t v = (uint8_t)b.take(3);
            if (lane == 0) h.lens[c_clorder[i]] = v;
        }
        __syncwarp();
        if (build_code(h.lens, 19, h.lcount, h.lsym, nullptr, 0, lane) != 0) return BGZF_BAD_CODE_LENGTHS;
        // the code-length code is decoded from lsym / lcount; the lengths themselves go to lens[] (registers first)
        int idx = 0;
        while (idx < nlen + ndist) {
            b.refill();
            int l = 0;
            const int s = slow_decode(b, h.lcount, h.lsym, l);
            if (s < 0) return BGZF_BAD_CODE;
            b.drop(l);
            int rep = 1;
            uint8_t v = (uint8_t)s;
            if (s == 16) {
                if (idx == 0) return BGZF_BAD_CODE_LENGTHS;
                __syncwarp();
                v = h.lens[idx - 1];
                rep = 3 + (int)b.take(2);
            } else if (s == 17) { v = 0; rep = 3 + (int)b.take(3); }
            else if (s == 18) { v = 0; rep = 11 + (int)b.take(7); }
            if (idx + rep > nlen + ndist) return BGZF_BAD_CODE_LENGTHS;
            __syncwarp();
            if (lane == 0) for (int i = 0; i < rep; ++i) h.lens[idx + i] = v;
            idx += rep;
        }
        if (b.overrun()) return BGZF_TRUNCATED;
        __syncwarp();
        if (h.lens[256] == 0) return BGZF_BAD_CODE_LENGTHS;
        // lens[nlen ..] moves to lens[288 ..] so that the two codes sit where the fixed ones do
        uint8_t dl = lane < ndist ? h.lens[nlen + lane] : 0;
        __syncwarp();
        h.lens[288 + lane] = dl;
        __syncwarp();
        build_code(h.lens, nlen, h.lcount, h.lsym, h.lfast, kLitFast, lane);
        if (!code_usable(h.lcount, nlen)) return BGZF_BAD_CODE_LENGTHS;
        build_code(h.lens + 288, ndist, h.dcount, h.dsym, h.dfast, kDistFast, lane);
        if (!code_usable(h.dcount, ndist)) return BGZF_BAD_CODE_LENGTHS;
    }
    // the compressed data of the block: at most 15 + 5 + 15 + 13 = 48 bits per symbol, one refill each
    for (;;) {
        b.refill();
        // a gzip range reads zeros past the end of its piece's data: stop there rather than decode them until the output is full
        if constexpr (sizeof(T) == 2) {
            if (b.overrun()) return BGZF_TRUNCATED;
        }
        int s = decode(b, h.lfast, kLitFast, h.lcount, h.lsym);
        if (s < 0) return BGZF_BAD_CODE;
        if (s < 256) {
            if (op >= out_len) return BGZF_OUTPUT_OVERFLOW;
            if (lane == 0) out[op] = (T)s;
            ++op;
            continue;
        }
        if (s == 256) break;
        s -= 257;
        if (s >= 29) return BGZF_BAD_CODE;
        const u32 len = c_lbase[s] + b.take(c_lext[s]);
        const int d = decode(b, h.dfast, kDistFast, h.dcount, h.dsym);
        if (d < 0 || d >= 30) return BGZF_BAD_CODE;
        const u32 dist = c_dbase[d] + b.take(c_dext[d]);
        if (dist > op - lo && !markers) return BGZF_DISTANCE;
        if ((u64)op + len > out_len) return BGZF_OUTPUT_OVERFLOW;
        __syncwarp();                                  // literals of lane 0 visible to the warp
        // an overlapping copy (dist < len) repeats the dist bytes before op: out[op + t] = out[op - dist + t mod dist]
        if constexpr (sizeof(T) == 1) {
            for (u32 t = lane; t < len; t += 32) out[op + t] = out[op - dist + (dist >= len ? t : t % dist)];
        } else {
            if (dist > op) jmin = min(jmin, kWindow + op - dist);
            for (u32 t = lane; t < len; t += 32) {
                const long long q = (long long)op - dist + (dist >= len ? t : t % dist);
                out[op + t] = q >= 0 ? out[q] : (T)(kMarker | (u32)(kWindow + q));
            }
        }
        op += len;
        __syncwarp();
    }
    return 0;
}

}  // namespace infl
}  // namespace sg
