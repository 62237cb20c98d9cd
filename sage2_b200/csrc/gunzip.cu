// gunzip.cu -- ordinary (single-member or concatenated) gzip inflated on the device (DESIGN.md section 4b).
// A gzip stream does not say where its DEFLATE blocks begin, so a piece of it is cut speculatively, as rapidgzip and pugz do:
//
//   1. Block-start search: the piece's compressed bytes are cut into chunks of kChunk bytes, and every bit offset of every
//      chunk but the first is tested, one thread each, for a dynamic-Huffman block header that passes every check the
//      decoder makes (dynamic_header_ok).  The lowest offset per chunk is a candidate; a chunk without one merges into the
//      chunk before it.
//   2. Range decode: one warp per candidate runs the decoder of inflate.cuh from there until a block starts exactly at a
//      later candidate (a block boundary that passes a candidate without meeting it shows that candidate to be false), until
//      its output would overflow (it stops early at the block's start), or until the compressed bytes run out.  Symbols
//      are 16 bits: a back-reference before the range's first byte is a marker naming its place in the unknown 32 KiB
//      window.  A final block is followed by the trailer and either the next member's header (decoding goes on with an empty
//      window) or the end of the stream (anything but a gzip header, which zlib ignores).
//   3. Confirmation (host): the first range starts at the carried boundary; a range is confirmed when the confirmed range
//      before it stopped exactly at its start.  Candidates passed over are dropped; a range that stopped early leaves a gap
//      that a further pass decodes from the boundary where it stopped, until the piece is covered.  An error counts only
//      once its range is confirmed: ranges from false candidates often fail.  Ranges past the text bound are dropped and
//      start the next piece.
//   4. Stitch: the windows of the confirmed ranges are resolved in order from the text before them (one block), then every
//      marker is replaced in parallel and the text lands contiguously after the host prefix, where parse.cu's splitter
//      takes it.  Every member's CRC32 and ISIZE are checked over the resolved text (tile CRCs folded with crc32_combine on
//      the host); a member may span pieces, so its running CRC and length travel in the state with its last 32 KiB.
#include <string.h>
#include <algorithm>
#include <map>
#include "../../include/sage2gpu.h"
#include "inflate.cuh"

namespace sg {

namespace {

using namespace infl;

// compressed bytes per block-start chunk.  zlib's blocks on FASTQ are some 16-20 KB compressed (median at levels 6 / 1), so a
// chunk of 16 KiB finds about one block start each: one range per block, and a range's text (some 30-35 KB) far below its
// share of the output pool.  The search tests every bit whatever the chunk size.
constexpr u32 kChunk = 16 << 10;
constexpr int kEvents = 32;             // member ends / starts one range may meet before it stops early
constexpr int kWarps = 4;               // ranges in flight per block
constexpr u32 kTile = 64 << 10;         // text bytes per CRC tile
constexpr u32 kNeedMore = 0xFFFFu;      // parse_gzip_header: the header runs past the data
constexpr u64 kNoOffset = ~0ull;
constexpr u64 kMaxPool = 1ull << 32;    // symbols of a pass's output pool at most (8 GiB)

enum : u32 { END_MET = 1, END_EARLY, END_RANOUT, END_STREAM, END_ERROR };
enum : u32 { EV_END = 0, EV_START = 1 };

struct GzEvent {
    u32 kind, pos;      // EV_END: the member's text ends at symbol `pos` of the range; EV_START: the next one starts there
    u32 crc, isize;     // EV_END: the trailer
    u64 hoff;           // EV_START: byte offset of the member's header in the piece
};

struct GzRange {
    // set by the host
    u64 start;                  // bit offset in the piece
    uint16_t *out;              // out[0, out_cap): the range's symbols
    u32 out_cap, header, target;    // header: starts at a gzip member header; target: first candidate a block start may meet
    // set by the decoder
    u32 kind, meet, err, n_ev, out_len, jmin;   // jmin: lowest window position a marker names (kWindow: none)
    u32 stop_header;            // the boundary it stopped at is between members
    u64 stop;                   // bit offset of that boundary
    u64 err_off, jmin_off;      // byte offset of the block / member of the error, of the block that wrote the marker jmin
    GzEvent ev[kEvents];
};

__device__ __forceinline__ u32 le32(const uint8_t *p) { return (u32)p[0] | (u32)p[1] << 8 | (u32)p[2] << 16 | (u32)p[3] << 24; }

// The gzip member header at in[p, n) (magic already seen): 0 and its length, kNeedMore, GZIP_HEADER or GZIP_HEADER_CRC -- the
// checks of zlib's inflate (method 8, no reserved flag, FHCRC = the low 16 bits of the header's CRC32)
__device__ u32 parse_gzip_header(const uint8_t *in, u32 n, u32 p, u32 &len, const u32 *table)
{
    if ((u64)p + 10 > n) return kNeedMore;
    if (in[p + 2] != 8 || (in[p + 3] & 0xE0)) return GZIP_HEADER;
    const u32 flg = in[p + 3];
    u64 h = p + 10;
    if (flg & 4) {
        if (h + 2 > n) return kNeedMore;
        h += 2 + ((u32)in[h] | (u32)in[h + 1] << 8);
        if (h > n) return kNeedMore;
    }
    for (u32 f = 8; f <= 16; f <<= 1) {                 // FNAME, FCOMMENT: zero-terminated
        if (!(flg & f)) continue;
        while (h < n && in[h]) ++h;
        if (h >= n) return kNeedMore;
        ++h;
    }
    if (flg & 2) {
        if (h + 2 > n) return kNeedMore;
        u32 c = 0xffffffffu;
        for (u64 i = p; i < h; ++i) c = table[(c ^ in[i]) & 0xff] ^ (c >> 8);
        if ((~c & 0xffffu) != ((u32)in[h] | (u32)in[h + 1] << 8)) return GZIP_HEADER_CRC;
        h += 2;
    }
    len = (u32)(h - p);
    return 0;
}

// one range (module comment, step 2); the whole warp, results written by lane 0
__device__ void decode_range(const uint8_t *in, u32 n, bool final, const u64 *cand, u32 ncand, GzRange &R, Huff &h, const u32 *table, int lane)
{
    uint16_t *out = R.out;
    Bits b{ in, n, (u32)(R.start >> 3), 0, 0ull };
    b.refill();
    b.drop((int)(R.start & 7));
    u32 op = 0, lo = 0, jmin = kWindow, t = R.target, n_ev = 0, kind = 0, meet = 0, err = 0;
    u64 stop = R.start, err_off = 0, jmin_off = 0, member = kNoOffset;
    bool header = R.header != 0, markers = !header, stop_header = header;
    for (;;) {
        if (header) {                                   // byte-aligned at a member boundary
            const u32 p = (u32)(b.taken() >> 3);
            stop = 8ull * p;
            stop_header = true;
            if (n - p < 2) { kind = final ? END_STREAM : END_RANOUT; break; }
            if (in[p] != 0x1f || in[p + 1] != 0x8b) { kind = END_STREAM; break; }
            if (n_ev + 2 > (u32)kEvents) { kind = END_EARLY; break; }
            u32 hl = 0;
            const u32 e = parse_gzip_header(in, n, p, hl, table);
            if (e == kNeedMore && !final) { kind = END_RANOUT; break; }
            if (e) { kind = END_ERROR; err = e == kNeedMore ? (u32)BGZF_TRUNCATED : e; err_off = p; break; }
            if (lane == 0) R.ev[n_ev] = GzEvent{ EV_START, op, 0, 0, p };
            ++n_ev;
            b.seek(p + hl);
            b.refill();
            lo = op; markers = false; header = false; member = p;
        }
        const u64 blk = b.taken();
        stop = blk;
        stop_header = false;
        while (t < ncand && cand[t] < blk) ++t;
        if (t < ncand && cand[t] == blk) { kind = END_MET; meet = t; break; }
        const u32 op0 = op, jmin0 = jmin;
        const u64 jmin_off0 = jmin_off;
        b.refill();
        const bool last = b.take(1) != 0;
        const u32 e = inflate_block(b, h, out, op, R.out_cap, lo, markers, jmin, lane);
        // the data ran out inside the block: bits past the end taken, or a stored block longer than the bytes left (whose
        // LEN / NLEN were still inside)
        const bool over = b.overrun() || e == BGZF_TRUNCATED;
        if ((e == BGZF_OUTPUT_OVERFLOW && !over) || (over && !final)) {     // stop at the block's start
            kind = over ? END_RANOUT : END_EARLY;
            op = op0; jmin = jmin0;
            break;
        }
        if (e || over) { kind = END_ERROR; err = over ? (u32)BGZF_TRUNCATED : e; err_off = blk >> 3; break; }
        if (jmin < jmin0) jmin_off = blk >> 3;
        if (last) {                                     // the trailer, byte-aligned
            b.drop(b.cnt & 7);
            const u32 q = (u32)(b.taken() >> 3);
            if ((u64)q + 8 > n) {
                if (!final) { kind = END_RANOUT; op = op0; jmin = jmin0; jmin_off = jmin_off0; break; }
                kind = END_ERROR; err = BGZF_TRUNCATED; err_off = member; break;
            }
            if (lane == 0) R.ev[n_ev] = GzEvent{ EV_END, op, le32(in + q), le32(in + q + 4), member };
            ++n_ev;
            b.seek(q + 8);
            header = true;
        }
    }
    __syncwarp();
    if (lane == 0) {
        R.kind = kind; R.meet = meet; R.err = err; R.n_ev = n_ev; R.out_len = op; R.jmin = jmin;
        R.stop_header = stop_header ? 1 : 0; R.stop = stop; R.err_off = err_off; R.jmin_off = jmin_off;
    }
}

__global__ void __launch_bounds__(32 * kWarps) gzip_ranges_kernel(const uint8_t *__restrict__ in, u32 n, int final, const u64 *__restrict__ cand,
                                                                  u32 ncand, GzRange *__restrict__ rg, u32 nr)
{
    __shared__ u32 table[256], x2n[32];
    __shared__ Huff huff[kWarps];
    crc_tables(table, x2n);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (u32 r = blockIdx.x * kWarps + w; r < nr; r += gridDim.x * kWarps) decode_range(in, n, final != 0, cand, ncand, rg[r], huff[w], table, lane);
}

// Does a dynamic-Huffman block header that the decoder accepts start at bit `bit` of in[0, n)?  The checks of inflate_block
// in the order of their cost: BTYPE, HLIT / HDIST, a complete code-length code, run-length-coded lengths that decode to
// exactly HLIT + HDIST entries with no repeat first, a code for EOB, usable literal/length and distance codes.
__device__ bool dynamic_header_ok(const uint8_t *in, u32 n, u64 bit)
{
    Bits b{ in, n, (u32)(bit >> 3), 0, 0ull };
    b.refill();
    b.drop((int)(bit & 7));
    const u32 hd = b.peek(17);
    if (((hd >> 1) & 3) != 2) return false;
    const int nlen = (int)((hd >> 3) & 31) + 257, ndist = (int)((hd >> 8) & 31) + 1, ncode = (int)((hd >> 13) & 15) + 4;
    if (nlen > 286 || ndist > 30) return false;
    b.drop(17);
    b.refill();
    uint8_t cl[19] = {};
    uint16_t count[16] = {}, sym[19], offs[16];
    for (int i = 0; i < ncode; ++i) cl[c_clorder[i]] = (uint8_t)b.take(3);
    for (int s = 0; s < 19; ++s) count[cl[s]]++;
    if (code_left(count, 19) != 0) return false;
    offs[1] = 0;
    for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + count[l];
    for (int s = 0; s < 19; ++s) if (cl[s]) sym[offs[cl[s]]++] = (uint16_t)s;
    uint16_t lc[16] = {}, dc[16] = {};
    int idx = 0, prev = 0, len256 = 0;
    while (idx < nlen + ndist) {
        b.refill();
        int l = 0;
        const int s = slow_decode(b, count, sym, l);
        if (s < 0) return false;
        b.drop(l);
        int rep = 1, v = s;
        if (s == 16) {
            if (idx == 0) return false;
            v = prev; rep = 3 + (int)b.take(2);
        } else if (s == 17) { v = 0; rep = 3 + (int)b.take(3); }
        else if (s == 18) { v = 0; rep = 11 + (int)b.take(7); }
        if (idx + rep > nlen + ndist) return false;
        for (int i = 0; i < rep; ++i, ++idx) {
            if (idx < nlen) lc[v]++; else dc[v]++;
            if (idx == 256) len256 = v;
        }
        prev = v;
        if (b.overrun()) return false;
    }
    return len256 != 0 && code_usable(lc, nlen) && code_usable(dc, ndist);
}

__global__ void block_starts_kernel(const uint8_t *__restrict__ in, u32 n, unsigned long long *__restrict__ best)
{
    const u64 total = 8ull * n;
    for (u64 bit = 8ull * kChunk + (u64)blockIdx.x * blockDim.x + threadIdx.x; bit < total; bit += (u64)gridDim.x * blockDim.x)
        if (dynamic_header_ok(in, n, bit)) atomicMin(&best[bit / (8ull * kChunk)], (unsigned long long)bit);
}

// the window W[k] before confirmed range k (k = 1 .. K-1): the 32 KiB before range k-1's end, from W[k-1] and range k-1's
// symbols; W[0] is the carried window.  One block, in chain order.
__global__ void __launch_bounds__(1024) gzip_windows_kernel(uint16_t *const *__restrict__ outs, const u32 *__restrict__ lens, u32 K, uint8_t *W)
{
    for (u32 k = 1; k < K; ++k) {
        const uint8_t *pw = W + (u64)(k - 1) * kWindow;
        uint8_t *w = W + (u64)k * kWindow;
        const uint16_t *o = outs[k - 1];
        const u32 L = lens[k - 1];
        for (u32 j = threadIdx.x; j < kWindow; j += blockDim.x) {
            uint8_t v;
            if ((u64)j + L >= kWindow) {
                const u32 s = o[L - kWindow + j];
                v = s & kMarker ? pw[s & (kWindow - 1)] : (uint8_t)s;
            } else v = pw[j + L];
            w[j] = v;
        }
        __syncthreads();
    }
}

// every symbol of confirmed range blockIdx.y to its byte of the text
__global__ void gzip_replace_kernel(uint16_t *const *__restrict__ outs, const u32 *__restrict__ lens, const u64 *__restrict__ text_off,
                                    const uint8_t *__restrict__ W, uint8_t *__restrict__ text)
{
    const u32 k = blockIdx.y, L = lens[k];
    const uint16_t *o = outs[k];
    const uint8_t *w = W + (u64)k * kWindow;
    uint8_t *t = text + text_off[k];
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < L; i += gridDim.x * blockDim.x) {
        const u32 s = o[i];
        t[i] = s & kMarker ? w[s & (kWindow - 1)] : (uint8_t)s;
    }
}

struct Tile {
    u64 off;
    u32 len, member;
};

__global__ void __launch_bounds__(32 * kWarps) crc_tiles_kernel(const uint8_t *__restrict__ text, const Tile *__restrict__ tiles, u32 n, u32 *__restrict__ crc)
{
    __shared__ u32 table[256], x2n[32];
    crc_tables(table, x2n);
    const int lane = threadIdx.x & 31;
    for (u32 i = blockIdx.x * kWarps + (threadIdx.x >> 5); i < n; i += gridDim.x * kWarps) {
        const u32 c = warp_crc32(text + tiles[i].off, tiles[i].len, table, x2n, lane);
        if (lane == 0) crc[i] = c;
    }
}

// zlib's crc32_combine on the host
u32 crc32_combine_host(u32 crc1, u32 crc2, u64 len2)
{
    static const struct X2n {
        u32 v[32];
        X2n() { u32 p = 1u << 30; v[0] = p; for (int k = 1; k < 32; ++k) v[k] = p = multmodp(p, p); }
    } x2n;
    return multmodp(x2nmodp(x2n.v, len2, 3), crc1) ^ crc2;
}

// CUDA events around the kernels of a piece, summed
struct KernelClock {
    cudaEvent_t a = nullptr, b = nullptr;
    cudaStream_t st;
    float ms = 0;
    explicit KernelClock(cudaStream_t s) : st(s) { SG_CUDA(cudaEventCreate(&a)); SG_CUDA(cudaEventCreate(&b)); }
    ~KernelClock() { cudaEventDestroy(a); cudaEventDestroy(b); }
    void begin() { SG_CUDA(cudaEventRecord(a, st)); }
    void end()                                          // the stream is synchronised after the copies that follow
    {
        SG_CUDA(cudaEventRecord(b, st));
        SG_CUDA(cudaEventSynchronize(b));
        float t = 0;
        SG_CUDA(cudaEventElapsedTime(&t, a, b));
        ms += t;
    }
};

struct Member {
    u64 hoff;           // header offset in the file
    u32 crc0;           // CRC32 and text before this piece
    u64 len0;
    bool ended = false;
    u32 crc = 0, isize = 0;
};

}  // namespace

GzipPiece stage_inflate_gzip_piece(Context &c, const uint8_t *h_in, u64 n, bool final, u64 text_bound, void *state, const uint8_t *prefix,
                                   u64 prefix_bytes, DevBuf<uint8_t> &d_text)
{
    sage2gpu_gzip_state &S = *(sage2gpu_gzip_state *)state;
    cudaStream_t st = c.stream;
    SG_CHECK(current_arena(), "stage_inflate_gzip_piece needs the caller's ArenaScope (d_text lives in it)");
    SG_CHECK(n < 0xFFFF0000ull, "gzip pieces must be smaller than 4 GiB");
    SG_CHECK(S.bit < 8 && S.window_bytes <= kWindow && (S.in_member || S.bit == 0), "malformed gzip state");
    GzipPiece res;
    auto with_prefix = [&](u64 text) {
        d_text.alloc(prefix_bytes + text + 1, st);
        if (prefix_bytes) SG_CUDA(cudaMemcpyAsync(d_text.p, prefix, prefix_bytes, cudaMemcpyHostToDevice, st));
    };
    if (S.done) {                                       // after the stream's end everything is ignored, as zlib does
        with_prefix(0);
        res.in_consumed = n;
        S.offset += n;
        return res;
    }
    if (n == 0) {
        if (final && S.in_member) throw GzipError(S.member_offset, BGZF_TRUNCATED);
        S.done = final ? 1 : 0;
        with_prefix(0);
        return res;
    }
    KernelClock clock(st);
    DevBuf<uint8_t> d_in(n, st);
    SG_CUDA(cudaMemcpyAsync(d_in.p, h_in, n, cudaMemcpyHostToDevice, st));

    // 1. block-start candidates; cand[0] is the carried boundary
    std::vector<u64> cand{ S.bit };
    if (n > kChunk) {
        const u64 nchunks = (n + kChunk - 1) / kChunk;
        DevBuf<unsigned long long> d_best(nchunks, st);
        std::vector<unsigned long long> best(nchunks);
        SG_CUDA(cudaMemsetAsync(d_best.p, 0xFF, nchunks * sizeof(unsigned long long), st));
        clock.begin();
        block_starts_kernel<<<(unsigned)std::min<u64>((8ull * n + 255) / 256, (u64)kSMs * 32), 256, 0, st>>>(d_in.p, (u32)n, d_best.p);
        SG_LAUNCHED();
        clock.end();
        SG_CUDA(cudaMemcpyAsync(best.data(), d_best.p, nchunks * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        SG_CUDA(cudaStreamSynchronize(st));
        for (unsigned long long x : best) if (x != ~0ull) cand.push_back(x);
    }
    const u32 ncand = (u32)cand.size();
    DevBuf<u64> d_cand(ncand, st);
    SG_CUDA(cudaMemcpyAsync(d_cand.p, cand.data(), ncand * sizeof(u64), cudaMemcpyHostToDevice, st));

    // 2. ranges: one per candidate, then the gaps behind ranges that stopped early, pass after pass
    std::vector<GzRange> R(ncand);
    for (u32 i = 0; i < ncand; ++i) {
        memset(&R[i], 0, sizeof(GzRange));
        R[i].start = cand[i];
        R[i].header = i == 0 && !S.in_member;
        R[i].target = i + 1;
    }
    std::vector<u32> todo(ncand);
    for (u32 i = 0; i < ncand; ++i) todo[i] = i;
    std::map<std::pair<u64, u32>, u32> gap_of;          // (boundary, between members) -> the range decoded from there
    std::vector<DevBuf<uint16_t>> pools;
    u64 pool_syms = 2 * std::max<u64>(text_bound, 1 << 16);
    while (!todo.empty()) {
        const u64 cap = std::min<u64>(pool_syms / todo.size(), 0x7FFFFFFFull);
        pools.emplace_back(cap * todo.size(), st);
        std::vector<GzRange> batch(todo.size());
        for (size_t j = 0; j < todo.size(); ++j) {
            GzRange &g = R[todo[j]];
            g.out = pools.back().p + j * cap;
            g.out_cap = (u32)cap;
            batch[j] = g;
        }
        DevBuf<GzRange> d_r(batch.size(), st);
        SG_CUDA(cudaMemcpyAsync(d_r.p, batch.data(), batch.size() * sizeof(GzRange), cudaMemcpyHostToDevice, st));
        const u64 blocks = (batch.size() + kWarps - 1) / kWarps;
        clock.begin();
        gzip_ranges_kernel<<<(unsigned)std::min<u64>(blocks, (u64)kSMs * 64), 32 * kWarps, 0, st>>>(d_in.p, (u32)n, final ? 1 : 0, d_cand.p, ncand, d_r.p,
                                                                                                     (u32)batch.size());
        SG_LAUNCHED();
        clock.end();
        SG_CUDA(cudaMemcpyAsync(batch.data(), d_r.p, batch.size() * sizeof(GzRange), cudaMemcpyDeviceToHost, st));
        SG_CUDA(cudaStreamSynchronize(st));
        res.ranges += batch.size();
        std::vector<u32> next;
        for (size_t j = 0; j < todo.size(); ++j) {
            const u32 i = todo[j];
            R[i] = batch[j];
            if (R[i].kind != END_EARLY) continue;
            if (R[i].out_len == 0 && R[i].n_ev == 0) {  // one block is more than its share of the pool: again with a larger pool
                if (pool_syms < kMaxPool) { pool_syms *= 2; next.push_back(i); }
                continue;
            }
            const std::pair<u64, u32> key{ R[i].stop, R[i].stop_header };
            if (gap_of.count(key)) continue;
            GzRange g;
            memset(&g, 0, sizeof(g));
            g.start = key.first;
            g.header = key.second;
            g.target = (u32)(std::upper_bound(cand.begin(), cand.end(), key.first) - cand.begin());
            gap_of[key] = (u32)R.size();
            next.push_back((u32)R.size());
            R.push_back(g);
        }
        todo.swap(next);
    }

    // 3. the confirmed chain from range 0, cut at the text bound (the first range is always taken)
    std::vector<u32> chain;
    u64 text = 0, cut = 0;
    u32 cut_header = 0;
    bool done = false;
    std::vector<Member> members;
    int m = -1;                                         // the open member
    if (S.in_member) { members.push_back(Member{ S.member_offset, S.crc, S.member_bytes }); m = 0; }
    for (u32 r = 0;;) {
        const GzRange &g = R[r];
        if (!chain.empty() && text + g.out_len > text_bound) { cut = g.start; cut_header = g.header; break; }
        if (g.kind == END_ERROR) {
            u64 off = g.err_off == kNoOffset ? (m >= 0 ? members[m].hoff : S.offset) : S.offset + g.err_off;
            throw GzipError(off, g.err);
        }
        chain.push_back(r);
        text += g.out_len;
        for (u32 e = 0; e < g.n_ev; ++e)
            if (g.ev[e].kind == EV_START) { members.push_back(Member{ S.offset + g.ev[e].hoff, 0, 0 }); m = (int)members.size() - 1; }
            else m = -1;
        if (g.kind == END_MET) { r = g.meet; continue; }
        if (g.kind == END_EARLY) {
            const auto gap = gap_of.find({ g.stop, g.stop_header });
            SG_CHECK(gap != gap_of.end(), "a DEFLATE block inflates to more than 4 GiB");
            r = gap->second;
            continue;
        }
        cut = g.stop;
        cut_header = g.stop_header;
        done = g.kind == END_STREAM;
        break;
    }
    std::vector<bool> confirmed(R.size(), false);
    for (u32 r : chain) confirmed[r] = true;
    for (u32 i = 1; i < ncand; ++i)
        if (cand[i] < cut && !confirmed[i]) ++res.rejected;
    res.confirmed = chain.size();

    // markers against the valid window (the member's text before each range), text offsets, member segments
    const u32 K = (u32)chain.size();
    SG_CHECK(K < 65535, "too many ranges in one gzip piece");
    std::vector<uint16_t *> outs(K);
    std::vector<u32> lens(K);
    std::vector<u64> toff(K);
    std::vector<Tile> tiles;
    u64 pos = 0, seg = 0;
    u32 avail = S.in_member ? S.window_bytes : 0;
    m = S.in_member ? 0 : -1;
    int mi = m;                                         // members[] index of the next START
    auto add_segment = [&](u64 a, u64 e, int mem) {
        for (u64 x = a; x < e; x += kTile) tiles.push_back(Tile{ prefix_bytes + x, (u32)std::min<u64>(kTile, e - x), (u32)mem });
    };
    for (u32 k = 0; k < K; ++k) {
        const GzRange &g = R[chain[k]];
        if (g.jmin < kWindow - avail) throw GzipError(S.offset + g.jmin_off, BGZF_DISTANCE);
        outs[k] = g.out;
        lens[k] = g.out_len;
        toff[k] = prefix_bytes + pos;
        long long last_start = -1;
        for (u32 e = 0; e < g.n_ev; ++e) {
            const u64 at = pos + g.ev[e].pos;
            if (g.ev[e].kind == EV_END) {
                SG_CHECK(m >= 0, "gzip trailer outside a member");
                add_segment(seg, at, m);
                members[m].ended = true;
                members[m].crc = g.ev[e].crc;
                members[m].isize = g.ev[e].isize;
                m = -1;
            } else {
                m = ++mi;
                seg = at;
                last_start = g.ev[e].pos;
            }
        }
        avail = (u32)(last_start >= 0 ? std::min<u64>(kWindow, g.out_len - last_start) : std::min<u64>(kWindow, (u64)avail + g.out_len));
        pos += g.out_len;
    }
    if (m >= 0) add_segment(seg, pos, m);

    // 4. windows, markers replaced, CRC tiles
    with_prefix(text);
    if (K) {
        DevBuf<uint8_t> d_w((u64)K * kWindow, st);
        DevBuf<uint16_t *> d_outs(K, st);
        DevBuf<u32> d_lens(K, st);
        DevBuf<u64> d_toff(K, st);
        SG_CUDA(cudaMemcpyAsync(d_w.p, S.window, kWindow, cudaMemcpyHostToDevice, st));
        SG_CUDA(cudaMemcpyAsync(d_outs.p, outs.data(), K * sizeof(uint16_t *), cudaMemcpyHostToDevice, st));
        SG_CUDA(cudaMemcpyAsync(d_lens.p, lens.data(), K * sizeof(u32), cudaMemcpyHostToDevice, st));
        SG_CUDA(cudaMemcpyAsync(d_toff.p, toff.data(), K * sizeof(u64), cudaMemcpyHostToDevice, st));
        const u32 longest = *std::max_element(lens.begin(), lens.end());
        clock.begin();
        gzip_windows_kernel<<<1, 1024, 0, st>>>(d_outs.p, d_lens.p, K, d_w.p);
        SG_LAUNCHED();
        if (longest) {
            gzip_replace_kernel<<<dim3((unsigned)std::min<u64>((longest + 4095) / 4096, 256), K), 256, 0, st>>>(d_outs.p, d_lens.p, d_toff.p, d_w.p, d_text.p);
            SG_LAUNCHED();
        }
        clock.end();
    }
    std::vector<u32> tcrc(tiles.size());
    if (!tiles.empty()) {
        DevBuf<Tile> d_tiles(tiles.size(), st);
        DevBuf<u32> d_crc(tiles.size(), st);
        SG_CUDA(cudaMemcpyAsync(d_tiles.p, tiles.data(), tiles.size() * sizeof(Tile), cudaMemcpyHostToDevice, st));
        clock.begin();
        crc_tiles_kernel<<<(unsigned)std::min<u64>((tiles.size() + kWarps - 1) / kWarps, (u64)kSMs * 16), 32 * kWarps, 0, st>>>(d_text.p, d_tiles.p,
                                                                                                                               (u32)tiles.size(), d_crc.p);
        SG_LAUNCHED();
        clock.end();
        SG_CUDA(cudaMemcpyAsync(tcrc.data(), d_crc.p, tiles.size() * sizeof(u32), cudaMemcpyDeviceToHost, st));
        SG_CUDA(cudaStreamSynchronize(st));
    }
    for (size_t i = 0; i < tiles.size(); ++i) {
        Member &x = members[tiles[i].member];
        x.crc0 = crc32_combine_host(x.crc0, tcrc[i], tiles[i].len);
        x.len0 += tiles[i].len;
    }
    for (const Member &x : members) {
        if (!x.ended) continue;
        if (x.crc0 != x.crc) throw GzipError(x.hoff, BGZF_CRC);
        if ((u32)x.len0 != x.isize) throw GzipError(x.hoff, BGZF_ISIZE);
    }

    // the state at the cut: the open member's CRC, length and last 32 KiB
    const u64 old = S.offset;
    S.offset += done ? n : cut >> 3;
    S.bit = cut_header || done ? 0 : (u32)(cut & 7);
    S.done = done ? 1 : 0;
    S.in_member = m >= 0 ? 1 : 0;
    if (m >= 0) {
        const Member &x = members[m];
        const u64 mine = pos - seg;                     // the open member's text in this piece
        const u64 keep = std::min<u64>(kWindow, mine);
        if (keep < kWindow) memmove(S.window, S.window + keep, kWindow - keep);
        if (keep) {
            SG_CUDA(cudaMemcpyAsync(S.window + kWindow - keep, d_text.p + prefix_bytes + pos - keep, keep, cudaMemcpyDeviceToHost, st));
            SG_CUDA(cudaStreamSynchronize(st));
        }
        S.member_offset = x.hoff;
        S.crc = x.crc0;
        S.member_bytes = x.len0;
        S.window_bytes = avail;
    } else {
        S.member_offset = S.crc = 0;
        S.member_bytes = 0;
        S.window_bytes = 0;
    }
    res.text_bytes = text;
    res.in_consumed = S.offset - old;
    res.kernel_ms = clock.ms;
    return res;
}

}  // namespace sg
