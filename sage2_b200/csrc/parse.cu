// parse.cu -- FASTA / FASTQ record splitting on the device (SURVEY.md 8(f) N2): the host only moves raw text.
// Restates what the reference does per record through kseq (inputReader/fastAQReader.cpp:16-45,
// readLoader.cpp:146-160) for the REGULAR layouts -- 4-line FASTQ (@name / sequence / +... / quality of the
// same length) and 2-line FASTA (>name / sequence).  Anything else (multi-line records, blank lines, a
// sequence line that starts with '>', '@' or '+', an empty sequence, a truncated tail) makes the call report
// "irregular" without appending anything, and the caller hands that text to its sequential parser.
//
// Per chunk: newline flags -> exclusive scan -> line starts; per record a structure check and the sequence
// length -> exclusive scan -> sequences copied (one warp per record) behind what was uploaded before.
#include <fcntl.h>
#include <string.h>
#include <sys/stat.h>
#include <unistd.h>
#include "context.h"

namespace sg {

__global__ void __launch_bounds__(256) nl_flag_kernel(const uint8_t *__restrict__ text, u64 n, u32 *__restrict__ flag)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) flag[i] = text[i] == '\n';
}

__global__ void __launch_bounds__(256) line_start_kernel(const uint8_t *__restrict__ text, u64 n, const u32 *__restrict__ idx, u32 *__restrict__ ls)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        if (i == 0) ls[0] = 0;
        if (text[i] == '\n') ls[idx[i] + 1] = (u32)(i + 1);
    }
}

// out[0] = bytes consumed by R records, out[1] |= 1 on any irregular record
__global__ void __launch_bounds__(256) record_check_kernel(const uint8_t *__restrict__ text, const u32 *__restrict__ ls, u64 R, int lpr, int marker,
                                                            u32 *__restrict__ seq_len, u32 *__restrict__ out)
{
    bool bad = false;
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (u64)gridDim.x * blockDim.x) {
        const u32 h0 = ls[lpr * r], s0 = ls[lpr * r + 1], s1 = ls[lpr * r + 2];
        bad |= text[h0] != (uint8_t)marker;
        u32 sl = s1 - 1 - s0;                                      // without the '\n'
        if (sl && text[s0 + sl - 1] == '\r') --sl;
        const uint8_t c0 = sl ? text[s0] : (uint8_t)'>';
        bad |= sl == 0 || c0 == '>' || c0 == '@' || c0 == '+';
        if (lpr == 4) {
            const u32 q0 = ls[4 * r + 3], q1 = ls[4 * r + 4];
            u32 ql = q1 - 1 - q0;
            if (ql && text[q0 + ql - 1] == '\r') --ql;
            bad |= text[s1] != '+' || ql != sl;
        }
        seq_len[r] = sl;
        if (r + 1 == R) out[0] = ls[lpr * R];
    }
    if (bad) atomicOr(&out[1], 1u);
}

__global__ void __launch_bounds__(256) record_copy_kernel(const uint8_t *__restrict__ text, const u32 *__restrict__ ls, const u32 *__restrict__ seq_len,
                                                           const u32 *__restrict__ seq_off, u64 R, int lpr, u64 base_off,
                                                           uint8_t *__restrict__ bases, int64_t *__restrict__ offsets)
{
    const int lane = threadIdx.x & 31;
    const u64 nwarps = (u64)gridDim.x * (blockDim.x >> 5);
    for (u64 r = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < R; r += nwarps) {
        const u32 s0 = ls[lpr * r + 1], sl = seq_len[r];
        const u64 o = base_off + seq_off[r];
        for (u32 t = lane; t < sl; t += 32) bases[o + t] = text[s0 + t];
        if (lane == 0) { offsets[r] = (int64_t)o; if (r + 1 == R) offsets[R] = (int64_t)(o + sl); }
    }
}

template <typename T>
static void grow_persistent(DevBuf<T> &b, size_t used, size_t need, cudaStream_t st)
{
    if (need <= b.cap) { b.n = need; return; }
    size_t cap = b.cap ? b.cap : (size_t)1 << 20;
    while (cap < need) cap += cap / 2 + 1;
    DevBuf<T> nb;
    nb.persistent = true;
    nb.alloc(cap, st);
    if (used) SG_CUDA(cudaMemcpyAsync(nb.p, b.p, used * sizeof(T), cudaMemcpyDeviceToDevice, st));
    b = std::move(nb);
}

static unsigned pgrid(u64 n, unsigned per_thread = 4)
{
    unsigned g = grid_for(n, 256, per_thread);
    return g > kSMs * 16u ? kSMs * 16u : g;
}

// The record splitter of both entries below: d_text[0, n_bytes) on the device, with room for one more byte; first / last = its
// first and last byte (the host knows them without a copy when the text came from the host)
static bool split_device_text(Context &c, uint8_t *d_text, u64 n_bytes, uint8_t first, uint8_t last, bool final, int &marker, u64 max_records,
                              u64 &consumed, u64 &n_records)
{
    cudaStream_t st = c.stream;
    if (marker == 0) {
        if (first != '@' && first != '>') return false;
        marker = first;
    }
    const int lpr = marker == '@' ? 4 : 2;
    const bool add_nl = final && last != '\n';
    const u64 n = n_bytes + (add_nl ? 1 : 0);
    if (add_nl) SG_CUDA(cudaMemsetAsync(d_text + n_bytes, '\n', 1, st));
    DevBuf<u32> flag(n, st), idx(n, st), d_lines(1, st);
    nl_flag_kernel<<<pgrid(n), 256, 0, st>>>(d_text, n, flag.p);
    SG_LAUNCHED();
    exclusive_scan_u32(flag.p, idx.p, n, d_lines.p, st);
    u32 L = 0;
    SG_CUDA(cudaMemcpyAsync(&L, d_lines.p, sizeof(u32), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    u64 R = (u64)L / (u64)lpr;
    if (R > max_records) R = max_records;
    if (R == 0) return !final;                       // no complete record in this chunk (a final stub is irregular)
    DevBuf<u32> ls((size_t)L + 1, st);
    line_start_kernel<<<pgrid(n), 256, 0, st>>>(d_text, n, idx.p, ls.p);
    SG_LAUNCHED();
    DevBuf<u32> seq_len(R, st), seq_off(R, st), d_out(3, st);
    SG_CUDA(cudaMemsetAsync(d_out.p, 0, 3 * sizeof(u32), st));
    record_check_kernel<<<pgrid(R, 1), 256, 0, st>>>(d_text, ls.p, R, lpr, marker, seq_len.p, d_out.p);
    SG_LAUNCHED();
    exclusive_scan_u32(seq_len.p, seq_off.p, R, d_out.p + 2, st);
    u32 h_out[3];
    SG_CUDA(cudaMemcpyAsync(h_out, d_out.p, sizeof(h_out), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    if (h_out[1]) return false;
    const u64 used = h_out[0], nb = h_out[2];
    if (final && R < max_records && used != n) return false;      // a truncated last record: let the sequential parser decide
    SG_CHECK(c.up_reads + R < 0x3FFFFFFFull, "at most 2^30-1 reads per context");
    grow_persistent(c.up_d_bases, (size_t)c.up_bases, (size_t)(c.up_bases + nb), st);
    grow_persistent(c.up_d_offsets, (size_t)(c.up_reads ? c.up_reads + 1 : 0), (size_t)(c.up_reads + R + 1), st);
    unsigned g = grid_for(R, 8, 1);
    if (g > kSMs * 16u) g = kSMs * 16u;
    record_copy_kernel<<<g, 256, 0, st>>>(d_text, ls.p, seq_len.p, seq_off.p, R, lpr, c.up_bases, c.up_d_bases.p, c.up_d_offsets.p + c.up_reads);
    SG_LAUNCHED();
    SG_CUDA(cudaStreamSynchronize(st));              // the caller may overwrite `text` now
    c.up_reads += R;
    c.up_bases += nb;
    consumed = used > n_bytes ? n_bytes : used;
    n_records = R;
    return true;
}

bool stage_parse_text_chunk(Context &c, const uint8_t *text, u64 n_bytes, bool final, int &marker, u64 max_records, u64 &consumed, u64 &n_records)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    consumed = 0; n_records = 0;
    if (n_bytes == 0 || max_records == 0) return true;
    SG_CHECK(n_bytes < 0x7FFFFFF0ull, "text chunks must be smaller than 2 GiB");
    DevBuf<uint8_t> d_text(n_bytes + 1, st);
    SG_CUDA(cudaMemcpyAsync(d_text.p, text, n_bytes, cudaMemcpyHostToDevice, st));
    return split_device_text(c, d_text.p, n_bytes, text[0], text[n_bytes - 1], final, marker, max_records, consumed, n_records);
}

bool stage_parse_device_text(Context &c, uint8_t *d_text, u64 n_bytes, bool final, int &marker, u64 max_records, u64 &consumed, u64 &n_records)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    consumed = 0; n_records = 0;
    if (n_bytes == 0 || max_records == 0) return true;
    SG_CHECK(n_bytes < 0x7FFFFFF0ull, "text chunks must be smaller than 2 GiB");
    uint8_t ends[2];
    SG_CUDA(cudaMemcpyAsync(&ends[0], d_text, 1, cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaMemcpyAsync(&ends[1], d_text + n_bytes - 1, 1, cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    return split_device_text(c, d_text, n_bytes, ends[0], ends[1], final, marker, max_records, consumed, n_records);
}

// drop the uploaded reads [first, first + count)
__global__ void __launch_bounds__(256) shift_offsets_kernel(const int64_t *__restrict__ in, u64 n, int64_t delta, int64_t *__restrict__ out)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) out[i] = in[i] - delta;
}

void stage_remove_uploaded(Context &c, u64 first, u64 count)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    SG_CHECK(first + count <= c.up_reads, "range outside the uploaded reads");
    if (count == 0) return;
    int64_t o[2];
    SG_CUDA(cudaMemcpyAsync(&o[0], c.up_d_offsets.p + first, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaMemcpyAsync(&o[1], c.up_d_offsets.p + first + count, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    const u64 tail_reads = c.up_reads - (first + count), tail_bases = c.up_bases - (u64)o[1];
    if (tail_reads) {
        DevBuf<uint8_t> tb(tail_bases, st);
        DevBuf<int64_t> to(tail_reads + 1, st);
        SG_CUDA(cudaMemcpyAsync(tb.p, c.up_d_bases.p + o[1], tail_bases, cudaMemcpyDeviceToDevice, st));
        SG_CUDA(cudaMemcpyAsync(c.up_d_bases.p + o[0], tb.p, tail_bases, cudaMemcpyDeviceToDevice, st));
        shift_offsets_kernel<<<pgrid(tail_reads + 1), 256, 0, st>>>(c.up_d_offsets.p + first + count, tail_reads + 1, o[1] - o[0], to.p);
        SG_LAUNCHED();
        SG_CUDA(cudaMemcpyAsync(c.up_d_offsets.p + first, to.p, (tail_reads + 1) * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
        SG_CUDA(cudaStreamSynchronize(st));
    }
    c.up_reads -= count;
    c.up_bases -= (u64)(o[1] - o[0]);
}

// ---- a saved .reads file: what ReadLoader::saveReadsInFile writes (readLoader.cpp:270-287), read back as
// ReadLoader::loadReadsFromFile does (readLoader.cpp:289).  Line 1 is the number of reads U, then one line per unique read
// "FREQ\tLEN\tF\tR\n".  Per piece of text: newline flags -> exclusive scan -> line starts (the kernels above); one warp per
// line parses and checks the fields; exclusive scan of the lengths; F copied (one warp per line) behind what was uploaded
// before, where the pack of step 1 takes it.  The order of the lines is checked after the pack (reads.cu).
enum SavedRule : u32 { SR_FREQ = 1, SR_LEN, SR_TOO_LONG, SR_SHORT, SR_LAYOUT, SR_F_CHAR, SR_R_CHAR, SR_REVCOMP, SR_CANON };

static std::string saved_rule_text(u32 r, int k)
{
    switch (r) {
        case SR_FREQ: return "FREQ is not a decimal in 0..65535 without leading zeros followed by a tab";
        case SR_LEN: return "LEN is not a decimal in 1..1016 without leading zeros followed by a tab";
        case SR_TOO_LONG: return "the read is longer than 1016 bases: not supported by this build of libsage2gpu";
        case SR_SHORT: return "the read is not longer than -k (" + std::to_string(k) + "): step 1 would have dropped it";
        case SR_LAYOUT: return "the line is not FREQ<tab>LEN<tab>F<tab>R with |F| = |R| = LEN";
        case SR_F_CHAR: return "F contains a character other than A, C, G, T";
        case SR_R_CHAR: return "R contains a character other than A, C, G, T";
        case SR_REVCOMP: return "R is not the reverse complement of F";
        case SR_CANON: return "F is not the canonical strand (F > R)";
        default: return "malformed line";
    }
}

__device__ __forceinline__ bool is_acgt(uint8_t ch) { return ch == 'A' || ch == 'C' || ch == 'G' || ch == 'T'; }
__device__ __forceinline__ uint8_t comp_base(uint8_t ch) { return ch == 'A' ? 'T' : ch == 'C' ? 'G' : ch == 'G' ? 'C' : ch == 'T' ? 'A' : 0; }

// a decimal without leading zeros at text[p, e), followed by a tab; false when malformed, else p moves past the tab
__device__ __forceinline__ bool saved_field(const uint8_t *text, u32 &p, u32 e, u32 &v)
{
    const u32 p0 = p;
    v = 0;
    while (p < e && p - p0 < 7 && text[p] >= '0' && text[p] <= '9') v = 10u * v + (u32)(text[p++] - '0');
    const u32 nd = p - p0;
    if (nd == 0 || nd >= 7 || (nd > 1 && text[p0] == '0') || p >= e || text[p] != '\t') return false;
    ++p;
    return true;
}

// one warp per line l (text[ls[l], ls[l+1]-1) + '\n'): seq_len / fstart = LEN and the offset of F (LEN 0 on a broken line), freq = FREQ;
// acc[0] = min(line << 8 | rule) over the broken lines, acc[1] = sum FREQ, acc[2] = sum FREQ * LEN, acc[3] = longest read
__global__ void __launch_bounds__(256) saved_line_kernel(const uint8_t *__restrict__ text, const u32 *__restrict__ ls, u64 L, int k, int max_ok,
                                                          u32 *__restrict__ seq_len, u32 *__restrict__ fstart, uint16_t *__restrict__ freq,
                                                          unsigned long long *__restrict__ acc)
{
    const int lane = threadIdx.x & 31;
    const u64 nwarps = (u64)gridDim.x * (blockDim.x >> 5);
    unsigned long long bad = ~0ull, sf = 0, sb = 0, mx = 0;
    for (u64 l = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); l < L; l += nwarps) {
        const u32 s = ls[l], e = ls[l + 1] - 1;
        u32 rule = 0, p = s, f = 0, n = 0;
        if (lane == 0) {
            if (!saved_field(text, p, e, f) || f > 65535u) rule = SR_FREQ;
            else if (!saved_field(text, p, e, n) || n == 0) rule = SR_LEN;
            else if (n > (u32)max_ok) rule = SR_TOO_LONG;
            else if ((int)n <= k) rule = SR_SHORT;
            else if (e - p != 2 * n + 1 || text[p + n] != '\t') rule = SR_LAYOUT;
        }
        rule = __shfl_sync(0xffffffffu, rule, 0);
        p = __shfl_sync(0xffffffffu, p, 0);
        n = __shfl_sync(0xffffffffu, n, 0);
        if (rule == 0) {
            const uint8_t *F = text + p, *R = F + n + 1;
            bool bf = false, br = false, mism = false;
            int order = 0;          // at the first position where F and R differ: 1 F < R, 2 F > R
            for (u32 b = 0; b < n; b += 32) {
                const u32 t = b + lane;
                uint8_t x = 0, y = 0;
                if (t < n) {
                    x = F[t]; y = R[t];
                    bf |= !is_acgt(x); br |= !is_acgt(y);
                    mism |= y != comp_base(F[n - 1 - t]);
                }
                const unsigned d = __ballot_sync(0xffffffffu, x != y);
                if (d && order == 0) order = __shfl_sync(0xffffffffu, x < y ? 1 : 2, __ffs(d) - 1);
            }
            if (__any_sync(0xffffffffu, bf)) rule = SR_F_CHAR;
            else if (__any_sync(0xffffffffu, br)) rule = SR_R_CHAR;
            else if (__any_sync(0xffffffffu, mism)) rule = SR_REVCOMP;
            else if (order == 2) rule = SR_CANON;
        }
        if (lane == 0) {
            seq_len[l] = rule ? 0u : n;
            fstart[l] = p;
            freq[l] = (uint16_t)f;
            if (rule) bad = min(bad, ((unsigned long long)l << 8) | rule);
            else { sf += f; sb += (unsigned long long)f * n; mx = max(mx, (unsigned long long)n); }
        }
    }
    if (lane == 0) {
        if (bad != ~0ull) atomicMin(&acc[0], bad);
        if (sf) atomicAdd(&acc[1], sf);
        if (sb) atomicAdd(&acc[2], sb);
        if (mx) atomicMax(&acc[3], mx);
    }
}

__global__ void __launch_bounds__(256) saved_copy_kernel(const uint8_t *__restrict__ text, const u32 *__restrict__ fstart, const u32 *__restrict__ seq_len,
                                                          const u32 *__restrict__ seq_off, u64 L, u64 base_off, uint8_t *__restrict__ bases,
                                                          int64_t *__restrict__ offsets)
{
    const int lane = threadIdx.x & 31;
    const u64 nwarps = (u64)gridDim.x * (blockDim.x >> 5);
    for (u64 l = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); l < L; l += nwarps) {
        const u32 s0 = fstart[l], sl = seq_len[l];
        const u64 o = base_off + seq_off[l];
        for (u32 t = lane; t < sl; t += 32) bases[o + t] = text[s0 + t];
        if (lane == 0) { offsets[l] = (int64_t)o; if (l + 1 == L) offsets[L] = (int64_t)(o + sl); }
    }
}

// the complete lines of text[0, n) (lines line0 + 1 .. of the slice) appended to the upload; returns the bytes they take
static u64 parse_saved_piece(Context &c, const uint8_t *text, u64 n, u64 line0, int &max_len)
{
    cudaStream_t st = c.stream;
    ArenaScope arena_scope(c.arena, st);
    const uint8_t *last_nl = (const uint8_t *)memrchr(text, '\n', n);
    if (!last_nl) return 0;
    const u64 used = (u64)(last_nl - text) + 1;
    DevBuf<uint8_t> d_text(used, st);
    SG_CUDA(cudaMemcpyAsync(d_text.p, text, used, cudaMemcpyHostToDevice, st));
    DevBuf<u32> flag(used, st), idx(used, st), d_lines(1, st);
    nl_flag_kernel<<<pgrid(used), 256, 0, st>>>(d_text.p, used, flag.p);
    SG_LAUNCHED();
    exclusive_scan_u32(flag.p, idx.p, used, d_lines.p, st);
    u32 L = 0;
    SG_CUDA(cudaMemcpyAsync(&L, d_lines.p, sizeof(u32), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    SG_CHECK(c.up_reads + L < 0x3FFFFFFFull, "at most 2^30-1 reads per context");
    DevBuf<u32> ls((size_t)L + 1, st);
    line_start_kernel<<<pgrid(used), 256, 0, st>>>(d_text.p, used, idx.p, ls.p);
    SG_LAUNCHED();
    grow_persistent(c.up_d_freq, (size_t)c.up_reads, (size_t)(c.up_reads + L), st);
    DevBuf<u32> seq_len(L, st), seq_off(L, st), fstart(L, st), d_tot(1, st);
    DevBuf<unsigned long long> acc(4, st);
    SG_CUDA(cudaMemsetAsync(acc.p, 0, 4 * sizeof(unsigned long long), st));
    SG_CUDA(cudaMemsetAsync(acc.p, 0xFF, sizeof(unsigned long long), st));
    unsigned g = grid_for(L, 8, 1);
    if (g > kSMs * 16u) g = kSMs * 16u;
    saved_line_kernel<<<g, 256, 0, st>>>(d_text.p, ls.p, L, c.min_overlap, 32 * kMaxWords - 8, seq_len.p, fstart.p, c.up_d_freq.p + c.up_reads, acc.p);
    SG_LAUNCHED();
    exclusive_scan_u32(seq_len.p, seq_off.p, L, d_tot.p, st);
    unsigned long long h_acc[4];
    u32 nb = 0;
    SG_CUDA(cudaMemcpyAsync(h_acc, acc.p, sizeof(h_acc), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaMemcpyAsync(&nb, d_tot.p, sizeof(u32), cudaMemcpyDeviceToHost, st));
    SG_CUDA(cudaStreamSynchronize(st));
    if (h_acc[0] != ~0ull) throw FormatError(line0 + (h_acc[0] >> 8) + 1, saved_rule_text((u32)(h_acc[0] & 0xFF), c.min_overlap), true);
    grow_persistent(c.up_d_bases, (size_t)c.up_bases, (size_t)(c.up_bases + nb), st);
    grow_persistent(c.up_d_offsets, (size_t)(c.up_reads ? c.up_reads + 1 : 0), (size_t)(c.up_reads + L + 1), st);
    saved_copy_kernel<<<g, 256, 0, st>>>(d_text.p, fstart.p, seq_len.p, seq_off.p, L, c.up_bases, c.up_d_bases.p, c.up_d_offsets.p + c.up_reads);
    SG_LAUNCHED();
    SG_CUDA(cudaStreamSynchronize(st));              // the caller may overwrite `text` now
    c.up_reads += L;
    c.up_bases += nb;
    c.sr_good += h_acc[1];
    c.sr_bp += h_acc[2];
    if ((int)h_acc[3] > max_len) max_len = (int)h_acc[3];
    return used;
}

namespace {
struct Fd {
    int fd;
    explicit Fd(const char *path) : fd(open(path, O_RDONLY)) { if (fd < 0) throw IoError(std::string("cannot open ") + path); }
    ~Fd() { close(fd); }
    size_t pread_all(void *buf, size_t n, u64 off) const
    {
        size_t got = 0;
        while (got < n) {
            const ssize_t r = pread(fd, (char *)buf + got, n - got, (off_t)(off + got));
            if (r < 0) throw IoError("cannot read a saved .reads file");
            if (r == 0) break;
            got += (size_t)r;
        }
        return got;
    }
};
}  // namespace

void saved_reads_header(const char *path, u64 &n_reads, u64 &body_offset, u64 &body_bytes)
{
    Fd f(path);
    struct stat sb;
    if (fstat(f.fd, &sb) != 0) throw IoError(std::string("cannot read ") + path);
    uint8_t h[16];
    const size_t n = f.pread_all(h, sizeof(h), 0);
    if (n >= 2 && h[0] == 0x1f && h[1] == 0x8b) throw FormatError(1, "a gzip file: saved reads are read as plain text only");
    size_t i = 0;
    u64 v = 0;
    while (i < n && i < 11 && h[i] >= '0' && h[i] <= '9') v = 10 * v + (u64)(h[i++] - '0');
    if (i == 0 || i > 10 || (i > 1 && h[0] == '0') || i >= n || h[i] != '\n')
        throw FormatError(1, "the first line is not the number of reads (a decimal without leading zeros)");
    if (v >= 0x3FFFFFFFull) throw FormatError(1, "more than 2^30-1 reads: not supported by this build of libsage2gpu");
    n_reads = v;
    body_offset = i + 1;
    body_bytes = (u64)sb.st_size - body_offset;
}

// Bytes of a text piece; SAGE2GPU_UPLOAD_PIECE_BYTES makes them smaller (tests), as in the host program
static size_t saved_piece_bytes()
{
    const char *e = getenv("SAGE2GPU_UPLOAD_PIECE_BYTES");
    const long long x = e ? atoll(e) : 0;
    return x >= 4096 ? (size_t)x : (size_t)32 << 20;
}

void stage_parse_saved_reads(Context &c, const char *path, u64 begin, u64 end, u64 &n_lines, int &max_len)
{
    u64 declared = 0, body_off = 0, body = 0;
    saved_reads_header(path, declared, body_off, body);
    Fd f(path);
    c.up_reads = c.up_bases = 0;
    c.sr_good = c.sr_bp = 0;
    n_lines = 0;
    max_len = 0;
    if (end > body) end = body;
    // The slice's text: from the first line that starts at or after `begin` to the end of the line that holds byte end-1
    // (its lines are those whose first byte lies in [begin, end)).  after_nl(pos) = 1 + the first '\n' at or after pos.
    std::vector<uint8_t> probe(1 << 16);
    auto after_nl = [&](u64 pos) {
        for (;;) {
            if (pos >= body) return body;
            const size_t got = f.pread_all(probe.data(), probe.size(), body_off + pos);
            if (got == 0) return body;
            const void *q = memchr(probe.data(), '\n', got);
            if (q) return pos + (u64)((const uint8_t *)q - probe.data()) + 1;
            pos += got;
        }
    };
    if (begin >= end) return;
    const u64 start = begin == 0 ? 0 : after_nl(begin - 1);
    const u64 stop = end >= body ? body : after_nl(end - 1);
    if (start >= stop) return;
    const size_t cap = saved_piece_bytes();
    uint8_t *buf = nullptr;
    SG_CUDA(cudaHostAlloc((void **)&buf, cap, cudaHostAllocDefault));
    try {
        u64 pos = start, have = 0;
        while (pos < stop || have) {
            const size_t want = (size_t)std::min<u64>(cap - have, stop - pos);
            const size_t got = f.pread_all(buf + have, want, body_off + pos);
            if (got != want) throw IoError(std::string("cannot read ") + path);
            pos += got;
            have += got;
            const bool final = pos == stop;
            const u64 lines_before = c.up_reads;
            const u64 used = parse_saved_piece(c, buf, have, lines_before, max_len);
            if (used == 0 && !final && have == cap)
                throw FormatError(c.up_reads + 1, "a line longer than " + std::to_string(cap) + " bytes", true);
            have -= used;
            if (have) memmove(buf, buf + used, have);
            if (final && have) throw FormatError(c.up_reads + 1, "the last line does not end with a newline (a truncated file?)", true);
        }
    } catch (...) {
        cudaFreeHost(buf);
        throw;
    }
    cudaFreeHost(buf);
    n_lines = c.up_reads;
}

}  // namespace sg
