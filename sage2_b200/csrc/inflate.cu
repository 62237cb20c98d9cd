// inflate.cu -- BGZF members inflated on the device (DESIGN.md section 4b, N2 ingest).
// BGZF (htslib's bgzip) is a series of ordinary gzip members of at most 64 KiB of text each; every member states its
// compressed size in a `BC` extra subfield (BSIZE) and its CRC32 and inflated size (ISIZE) in the trailer, and no
// back-reference crosses a member.  The host walks the headers (bgzf_scan_members) and the device inflates every member of
// a batch at once, each into its place in one contiguous text buffer (the prefix sum of the ISIZEs), where the record
// splitter of parse.cu takes it.
//
// Layout: one warp per member.  Every lane runs the same DEFLATE decoder (RFC 1951) in lockstep on the same bits -- the
// loads are broadcasts and the control flow stays uniform -- while the lanes share the work that has width: filling the
// Huffman lookup tables, match copies, stored blocks and the CRC32 of the member's output (per-lane segments combined with
// the shift operators of zlib's crc32_combine).  Every bound is checked before the access it guards: reads stay inside
// the member, writes inside its ISIZE, no distance reaches before the member's first output byte.  A member that breaks a
// rule gets an error code; the batch reports the first bad member.
#include <string.h>
#include "context.h"

namespace sg {

namespace {

constexpr int kLitFast = 10;            // bits of the first-level literal/length table
constexpr int kDistFast = 8;            // bits of the first-level distance table
constexpr int kWarps = 4;               // members in flight per block
constexpr u32 kPoly = 0xedb88320u;      // CRC-32 (reflected)

// per-warp Huffman state in shared memory: canonical codes as counts per length + symbols in code order (puff's form),
// and first-level tables of (symbol | length << 12) for codes of at most kLitFast / kDistFast bits (0: longer code)
struct Huff {
    uint16_t lfast[1 << kLitFast];
    uint16_t dfast[1 << kDistFast];
    uint16_t lsym[288], dsym[32];
    uint16_t lcount[16], dcount[16];
    uint8_t lens[288 + 32];
};

__constant__ uint16_t c_lbase[29] = { 3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258 };
__constant__ uint8_t c_lext[29] = { 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0 };
__constant__ uint16_t c_dbase[30] = { 1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769,
                                      1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577 };
__constant__ uint8_t c_dext[30] = { 0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13 };
__constant__ uint8_t c_clorder[19] = { 16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15 };

// LSB-first bit reader over in[0, end) (the member's DEFLATE data).  Bytes past `end` read as zeros and are never loaded;
// overrun() says whether the bits taken so far reach past `end`.
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

// count / sym of the code with lengths[0, n) (lane 0), then the first-level table (all lanes).  Returns puff's `left`:
// 0 complete (or no codes at all), < 0 over-subscribed, > 0 incomplete.
__device__ int build_code(const uint8_t *lengths, int n, uint16_t *count, uint16_t *sym, uint16_t *fast, int fast_bits, int lane)
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
    int left = 1;
    if (count[0] == n) left = 0;
    else {
        for (int l = 1; l < 16; ++l) {
            left <<= 1;
            left -= count[l];
            if (left < 0) break;
        }
    }
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
__device__ __forceinline__ u32 multmodp(u32 a, u32 b)
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

__device__ __forceinline__ u32 x2nmodp(const u32 *x2n, u64 n, int k)
{
    u32 p = 1u << 31;
    while (n) {
        if (n & 1) p = multmodp(x2n[k & 31], p);
        n >>= 1;
        ++k;
    }
    return p;
}

// CRC32 of out[0, n), the warp's lanes over contiguous segments, combined as crc32_combine does
__device__ u32 warp_crc32(const uint8_t *out, u32 n, const u32 *table, const u32 *x2n, int lane)
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

// one member: the DEFLATE stream of in[0, in_len) into out[0, out_len); returns 0 or a BgzfError code
__device__ u32 inflate_member(const uint8_t *in, u32 in_len, uint8_t *out, u32 out_len, Huff &h, int lane)
{
    Bits b{ in, in_len, 0, 0, 0ull };
    u32 op = 0;
    bool last = false;
    // bits past the end read as zeros: an error met there is a truncated member
    auto fail = [&](u32 code) { return b.overrun() ? (u32)BGZF_TRUNCATED : code; };
    while (!last) {
        b.refill();
        last = b.take(1) != 0;
        const u32 type = b.take(2);
        if (type == 3) return fail(BGZF_BLOCK_TYPE);
        if (type == 0) {                                   // stored: byte-aligned LEN, NLEN, LEN bytes
            b.drop(b.cnt & 7);
            const u32 len = b.take(16), nlen = b.take(16);
            if (b.overrun()) return BGZF_TRUNCATED;
            if (len != (~nlen & 0xffffu)) return fail(BGZF_STORED_LEN);
            const u32 src = (u32)(b.taken() >> 3);
            if ((u64)src + len > in_len) return BGZF_TRUNCATED;
            if ((u64)op + len > out_len) return fail(BGZF_OUTPUT_OVERFLOW);
            for (u32 t = lane; t < len; t += 32) out[op + t] = in[src + t];
            op += len;
            b.pos = src + len; b.cnt = 0; b.buf = 0;
            __syncwarp();
            continue;
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
            if (nlen > 286 || ndist > 30) return fail(BGZF_BAD_CODE_LENGTHS);
            b.refill();
            __syncwarp();
            if (lane < 19) h.lens[lane] = 0;
            __syncwarp();
            for (int i = 0; i < ncode; ++i) {
                const uint8_t v = (uint8_t)b.take(3);
                if (lane == 0) h.lens[c_clorder[i]] = v;
            }
            __syncwarp();
            if (build_code(h.lens, 19, h.lcount, h.lsym, nullptr, 0, lane) != 0) return fail(BGZF_BAD_CODE_LENGTHS);
            // the code-length code is decoded from lsym / lcount; the lengths themselves go to lens[] (registers first)
            int idx = 0;
            while (idx < nlen + ndist) {
                b.refill();
                int l = 0;
                const int s = slow_decode(b, h.lcount, h.lsym, l);
                if (s < 0) return fail(BGZF_BAD_CODE);
                b.drop(l);
                int rep = 1;
                uint8_t v = (uint8_t)s;
                if (s == 16) {
                    if (idx == 0) return fail(BGZF_BAD_CODE_LENGTHS);
                    __syncwarp();
                    v = h.lens[idx - 1];
                    rep = 3 + (int)b.take(2);
                } else if (s == 17) { v = 0; rep = 3 + (int)b.take(3); }
                else if (s == 18) { v = 0; rep = 11 + (int)b.take(7); }
                if (idx + rep > nlen + ndist) return fail(BGZF_BAD_CODE_LENGTHS);
                __syncwarp();
                if (lane == 0) for (int i = 0; i < rep; ++i) h.lens[idx + i] = v;
                idx += rep;
            }
            if (b.overrun()) return BGZF_TRUNCATED;
            __syncwarp();
            if (h.lens[256] == 0) return fail(BGZF_BAD_CODE_LENGTHS);
            // lens[nlen ..] moves to lens[288 ..] so that the two codes sit where the fixed ones do
            uint8_t dl = lane < ndist ? h.lens[nlen + lane] : 0;
            __syncwarp();
            h.lens[288 + lane] = dl;
            __syncwarp();
            // incomplete codes only as a single one-bit code (zlib's inflate_table accepts that one)
            int err = build_code(h.lens, nlen, h.lcount, h.lsym, h.lfast, kLitFast, lane);
            if (err < 0 || (err > 0 && nlen != h.lcount[0] + h.lcount[1])) return fail(BGZF_BAD_CODE_LENGTHS);
            err = build_code(h.lens + 288, ndist, h.dcount, h.dsym, h.dfast, kDistFast, lane);
            if (err < 0 || (err > 0 && ndist != h.dcount[0] + h.dcount[1])) return fail(BGZF_BAD_CODE_LENGTHS);
        }
        // the compressed data of the block: at most 15 + 5 + 15 + 13 = 48 bits per symbol, one refill each
        for (;;) {
            b.refill();
            int s = decode(b, h.lfast, kLitFast, h.lcount, h.lsym);
            if (s < 0) return fail(BGZF_BAD_CODE);
            if (s < 256) {
                if (op >= out_len) return fail(BGZF_OUTPUT_OVERFLOW);
                if (lane == 0) out[op] = (uint8_t)s;
                ++op;
                continue;
            }
            if (s == 256) break;
            s -= 257;
            if (s >= 29) return fail(BGZF_BAD_CODE);
            const u32 len = c_lbase[s] + b.take(c_lext[s]);
            const int d = decode(b, h.dfast, kDistFast, h.dcount, h.dsym);
            if (d < 0 || d >= 30) return fail(BGZF_BAD_CODE);
            const u32 dist = c_dbase[d] + b.take(c_dext[d]);
            if (dist > op) return fail(BGZF_DISTANCE);
            if ((u64)op + len > out_len) return fail(BGZF_OUTPUT_OVERFLOW);
            __syncwarp();                                  // literals of lane 0 visible to the warp
            // an overlapping copy (dist < len) repeats the dist bytes before op: out[op + t] = out[op - dist + t mod dist]
            for (u32 t = lane; t < len; t += 32) out[op + t] = out[op - dist + (dist >= len ? t : t % dist)];
            op += len;
            __syncwarp();
        }
        if (b.overrun()) return BGZF_TRUNCATED;
    }
    if (b.overrun()) return BGZF_TRUNCATED;
    if (((b.taken() + 7) >> 3) != in_len) return BGZF_TRAILING;     // the trailer follows the last block's final byte
    if (op != out_len) return BGZF_ISIZE;
    __syncwarp();
    return 0;
}

__global__ void __launch_bounds__(32 * kWarps) inflate_members_kernel(const uint8_t *__restrict__ in, const BgzfMember *__restrict__ mem, u64 n,
                                                                     uint8_t *__restrict__ out, unsigned long long *__restrict__ bad)
{
    __shared__ u32 table[256], x2n[32];
    __shared__ Huff huff[kWarps];
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
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (u64 m = (u64)blockIdx.x * kWarps + w; m < n; m += (u64)gridDim.x * kWarps) {
        const BgzfMember M = mem[m];
        const u32 data0 = M.header_bytes, data1 = M.in_bytes - 8;
        uint8_t *o = out + M.out_off;
        u32 err = inflate_member(in + M.in_off + data0, data1 - data0, o, M.out_bytes, huff[w], lane);
        if (!err && warp_crc32(o, M.out_bytes, table, x2n, lane) != M.crc) err = BGZF_CRC;
        if (err && lane == 0) atomicMin(bad, (unsigned long long)m << 8 | err);
    }
}

}  // namespace

const char *bgzf_error_text(u32 code)
{
    switch (code) {
        case BGZF_HEADER: return "not a gzip member with a BC (BSIZE) extra subfield";
        case BGZF_BSIZE: return "BSIZE reaches past the end of the data";
        case BGZF_ISIZE_LIMIT: return "ISIZE is larger than 65536";
        case BGZF_BLOCK_TYPE: return "DEFLATE block type 3";
        case BGZF_STORED_LEN: return "stored block LEN is not the one's complement of NLEN";
        case BGZF_BAD_CODE_LENGTHS: return "over-subscribed, incomplete or malformed Huffman code lengths";
        case BGZF_BAD_CODE: return "invalid Huffman code, literal/length or distance symbol";
        case BGZF_DISTANCE: return "a distance reaches before the member's first output byte";
        case BGZF_OUTPUT_OVERFLOW: return "more output than ISIZE";
        case BGZF_TRUNCATED: return "the DEFLATE data ends before its final block (truncated member)";
        case BGZF_TRAILING: return "the final block does not end at the member's trailer";
        case BGZF_ISIZE: return "less output than ISIZE";
        case BGZF_CRC: return "CRC32 of the output does not match the trailer";
        default: return "malformed member";
    }
}

// The header of the member at buf[off, n): its size (BSIZE + 1) and where its DEFLATE data starts.  0 = fine, else a
// BgzfError code.  FNAME / FCOMMENT / FHCRC are skipped as gzip readers skip them.
u32 bgzf_parse_header(const uint8_t *buf, u64 n, u64 off, u32 &member_bytes, u32 &header_bytes)
{
    const uint8_t *p = buf + off;
    const u64 avail = n - off;
    if (avail < 18 || p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4) || (p[3] & 0xE0)) return BGZF_HEADER;
    const u32 xlen = (u32)p[10] | (u32)p[11] << 8;
    if (12 + (u64)xlen > avail) return BGZF_HEADER;
    int bsize = -1;
    for (u32 i = 12; i + 4 <= 12 + xlen;) {
        const u32 slen = (u32)p[i + 2] | (u32)p[i + 3] << 8;
        if (i + 4 + slen > 12 + xlen) break;
        if (p[i] == 'B' && p[i + 1] == 'C' && slen == 2) bsize = (int)((u32)p[i + 4] | (u32)p[i + 5] << 8);
        i += 4 + slen;
    }
    if (bsize < 0) return BGZF_HEADER;
    member_bytes = (u32)bsize + 1;
    if (member_bytes > avail) return BGZF_BSIZE;
    u32 h = 12 + xlen;
    if (p[3] & 8) { while (h < member_bytes && p[h]) ++h; ++h; }      // FNAME
    if (p[3] & 16) { while (h < member_bytes && p[h]) ++h; ++h; }     // FCOMMENT
    if (p[3] & 2) h += 2;                                             // FHCRC
    if ((u64)h + 8 > member_bytes) return BGZF_HEADER;
    header_bytes = h;
    const uint8_t *t = p + member_bytes - 4;
    if (((u32)t[0] | (u32)t[1] << 8 | (u32)t[2] << 16 | (u32)t[3] << 24) > 65536u) return BGZF_ISIZE_LIMIT;
    return 0;
}

void bgzf_scan_members(const uint8_t *buf, u64 n, u64 out_base, std::vector<BgzfMember> &m, u64 &out_end)
{
    m.clear();
    u64 off = 0, o = out_base;
    while (off < n) {
        u32 mb = 0, hb = 0;
        if (const u32 e = bgzf_parse_header(buf, n, off, mb, hb)) throw BgzfError(m.size(), off, e);
        const uint8_t *t = buf + off + mb - 8;
        BgzfMember x;
        x.in_off = off;
        x.out_off = o;
        x.in_bytes = mb;
        x.header_bytes = hb;
        x.crc = (u32)t[0] | (u32)t[1] << 8 | (u32)t[2] << 16 | (u32)t[3] << 24;
        x.out_bytes = (u32)t[4] | (u32)t[5] << 8 | (u32)t[6] << 16 | (u32)t[7] << 24;
        m.push_back(x);
        off += mb;
        o += x.out_bytes;
    }
    out_end = o;
}

float stage_inflate_members(Context &c, const uint8_t *d_in, const BgzfMember *h_members, u64 n_members, uint8_t *d_out)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    if (n_members == 0) return 0.f;
    DevBuf<BgzfMember> d_mem(n_members, st);
    DevBuf<unsigned long long> d_bad(1, st);
    SG_CUDA(cudaMemcpyAsync(d_mem.p, h_members, n_members * sizeof(BgzfMember), cudaMemcpyHostToDevice, st));
    SG_CUDA(cudaMemsetAsync(d_bad.p, 0xFF, sizeof(unsigned long long), st));
    cudaEvent_t e0, e1;
    SG_CUDA(cudaEventCreate(&e0));
    SG_CUDA(cudaEventCreate(&e1));
    const u64 blocks = (n_members + kWarps - 1) / kWarps;
    SG_CUDA(cudaEventRecord(e0, st));
    inflate_members_kernel<<<(unsigned)std::min<u64>(blocks, (u64)kSMs * 64), 32 * kWarps, 0, st>>>(d_in, d_mem.p, n_members, d_out, d_bad.p);
    SG_LAUNCHED();
    SG_CUDA(cudaEventRecord(e1, st));
    unsigned long long bad = 0;
    SG_CUDA(cudaMemcpyAsync(&bad, d_bad.p, sizeof(bad), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (bad != ~0ull) {
        const u64 i = bad >> 8;
        throw BgzfError(i, h_members[i].in_off, (u32)(bad & 0xFF));
    }
    return ms;
}

}  // namespace sg
