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
#include "inflate.cuh"

namespace sg {

namespace {

using namespace infl;

constexpr int kWarps = 4;               // members in flight per block

// one member: the DEFLATE stream of in[0, in_len) into out[0, out_len); returns 0 or a BgzfError code
__device__ u32 inflate_member(const uint8_t *in, u32 in_len, uint8_t *out, u32 out_len, Huff &h, int lane)
{
    Bits b{ in, in_len, 0, 0, 0ull };
    u32 op = 0, jmin = kWindow;
    bool last = false;
    while (!last) {
        b.refill();
        last = b.take(1) != 0;
        // bits past the end read as zeros: an error met there is a truncated member
        if (const u32 err = inflate_block(b, h, out, op, out_len, 0, false, jmin, lane)) return b.overrun() ? (u32)BGZF_TRUNCATED : err;
        if (b.overrun()) return BGZF_TRUNCATED;
    }
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
    crc_tables(table, x2n);
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
        case GZIP_HEADER: return "malformed gzip member header (method, flags or a truncated header)";
        case GZIP_HEADER_CRC: return "the header CRC16 (FHCRC) does not match";
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
