// format.cu -- the reference's -s text files formatted on the device (SURVEY.md 8(f) N3).  Restates
// ReadLoader::saveReadsInFile / operator<<(Read) (inputReader/readLoader.cpp:29-36,270-287) and
// OverlapGraph::saveOverlapGraphInFile / operator<<(Edge*) (overlapGraph/overlapGraph.cpp:12-20,338-369)
// byte for byte, and the same graph as GFA 1.0 (no reference counterpart; format in include/sage2gpu.h).  Two passes per
// batch: line lengths -> exclusive scan -> every line written at its offset; the batch then leaves the device in one copy
// and the file in one fwrite.
#include <stdio.h>
#include "context.h"

namespace sg {

__device__ __forceinline__ int dec_digits(u32 v)
{
    return v < 10u ? 1 : v < 100u ? 2 : v < 1000u ? 3 : v < 10000u ? 4 : v < 100000u ? 5 : v < 1000000u ? 6
         : v < 10000000u ? 7 : v < 100000000u ? 8 : v < 1000000000u ? 9 : 10;
}
__device__ __forceinline__ char *put_dec(char *p, u32 v)
{
    const int n = dec_digits(v);
    for (int i = n - 1; i >= 0; --i) { p[i] = (char)('0' + v % 10u); v /= 10u; }
    return p + n;
}
__device__ __forceinline__ char *put_str(char *p, const char *s) { while (*s) *p++ = *s++; return p; }

// ---- <prefix>.graph3: per undirected edge "from\tto\ttype\t1\tdelta\t0\t0\n\n" and its twin ---------------
__device__ __forceinline__ void edge_fields(const u64 *edges, const uint16_t *len, u64 e, u32 &a, u32 &b, u32 &t, u32 &d, u32 &dt)
{
    const u64 w0 = edges[2 * e], w1 = edges[2 * e + 1];
    a = (u32)(w0 >> 32); b = (u32)w0;
    t = (u32)(w1 >> 20) & 3u; d = (u32)(w1 & 0xFFFFFu);
    dt = (u32)len[a - 1] - ((u32)len[b - 1] - d);            // overlapGraph.cpp:147
}

__global__ void __launch_bounds__(256) edge_len_kernel(const u64 *__restrict__ edges, const uint16_t *__restrict__ len, u64 e0, u64 n, u32 *__restrict__ out)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        u32 a, b, t, d, dt;
        edge_fields(edges, len, e0 + i, a, b, t, d, dt);
        out[i] = 2u * (u32)(dec_digits(a) + dec_digits(b)) + (u32)dec_digits(d) + (u32)dec_digits(dt) + 2u + 2u * 11u;
    }
}

__global__ void __launch_bounds__(256) edge_fmt_kernel(const u64 *__restrict__ edges, const uint16_t *__restrict__ len, u64 e0, u64 n,
                                                        const u32 *__restrict__ off, char *__restrict__ out)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        u32 a, b, t, d, dt;
        edge_fields(edges, len, e0 + i, a, b, t, d, dt);
        char *p = out + off[i];
        p = put_dec(p, a); *p++ = '\t'; p = put_dec(p, b); *p++ = '\t'; *p++ = (char)('0' + t);
        p = put_str(p, "\t1\t"); p = put_dec(p, d); p = put_str(p, "\t0\t0\n\n");
        p = put_dec(p, b); *p++ = '\t'; p = put_dec(p, a); *p++ = '\t'; *p++ = (char)('0' + reverse_edge_type(t));
        p = put_str(p, "\t1\t"); p = put_dec(p, dt); p = put_str(p, "\t0\t0\n\n");
    }
}

// ---- <prefix>.reads: per unique read "frequency\tlength\tFORWARD\tREVCOMP\n" ------------------------------
__global__ void __launch_bounds__(256) read_len_kernel(const uint16_t *__restrict__ len, const uint16_t *__restrict__ freq, u64 r0, u64 n, u32 *__restrict__ out)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        out[i] = (u32)dec_digits(freq[r0 + i]) + (u32)dec_digits(len[r0 + i]) + 2u * (u32)len[r0 + i] + 4u;
}

// one warp per read: lanes write the characters of both strands coalesced
__global__ void __launch_bounds__(256) read_fmt_kernel(const u64 *__restrict__ F, const u64 *__restrict__ RC, const uint16_t *__restrict__ len,
                                                        const uint16_t *__restrict__ freq, int SWS, u64 r0, u64 n,
                                                        const u32 *__restrict__ off, char *__restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const u64 nwarps = (u64)gridDim.x * (blockDim.x >> 5);
    for (u64 i = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += nwarps) {
        const u64 r = r0 + i;
        const u32 l = len[r], f = freq[r];
        char *p = out + off[i];
        const int hd = dec_digits(f) + dec_digits(l) + 2;
        if (lane == 0) { char *q = put_dec(p, f); *q++ = '\t'; q = put_dec(q, l); *q++ = '\t'; }
        char *s0 = p + hd, *s1 = s0 + l + 1;
        const u64 *fw = F + r * SWS, *rc = RC + r * SWS;
        for (u32 t = lane; t < l; t += 32) {
            const int sh = 62 - 2 * (int)(t & 31);
            s0[t] = "ACGT"[(fw[t >> 5] >> sh) & 3];
            s1[t] = "ACGT"[(rc[t >> 5] >> sh) & 3];
        }
        if (lane == 0) { s0[l] = '\t'; s1[l] = '\n'; }
    }
}

// ---- <prefix>.gfa: GFA 1.0 (include/sage2gpu.h, sage2gpu_write_gfa) --------------------------------------------
// per unique read "S\t<id>\t<F>\tLN:i:<len>\tRC:i:<freq>\n"
__global__ void __launch_bounds__(256) gfa_seg_len_kernel(const uint16_t *__restrict__ len, const uint16_t *__restrict__ freq, u64 r0, u64 n, u32 *__restrict__ out)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const u32 l = len[r0 + i];
        out[i] = (u32)dec_digits((u32)(r0 + i + 1)) + (u32)dec_digits(l) + (u32)dec_digits(freq[r0 + i]) + l + 16u;
    }
}

// one warp per read: lanes write the characters of F coalesced, as read_fmt_kernel does
__global__ void __launch_bounds__(256) gfa_seg_fmt_kernel(const u64 *__restrict__ F, const uint16_t *__restrict__ len, const uint16_t *__restrict__ freq,
                                                           int SWS, u64 r0, u64 n, const u32 *__restrict__ off, char *__restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const u64 nwarps = (u64)gridDim.x * (blockDim.x >> 5);
    for (u64 i = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += nwarps) {
        const u64 r = r0 + i;
        const u32 l = len[r], id = (u32)(r + 1);
        char *p = out + off[i];
        char *s = p + 2 + dec_digits(id) + 1;
        if (lane == 0) { *p++ = 'S'; *p++ = '\t'; p = put_dec(p, id); *p++ = '\t'; }
        const u64 *fw = F + r * SWS;
        for (u32 t = lane; t < l; t += 32) s[t] = "ACGT"[(fw[t >> 5] >> (62 - 2 * (int)(t & 31))) & 3];
        if (lane == 0) {
            char *q = put_str(s + l, "\tLN:i:"); q = put_dec(q, l);
            q = put_str(q, "\tRC:i:"); q = put_dec(q, freq[r]); *q = '\n';
        }
    }
}

// per undirected edge "L\t<a>\t<oa>\t<b>\t<ob>\t<n>M\n", n = len(b) - delta.  Orientations from the edge type (SURVEY 8 A8):
// 3 = fwd b prefix on fwd a suffix (+ +), 2 = rc b prefix on fwd a suffix (+ -), 0 = fwd b suffix on fwd a prefix (- -),
// 1 = rc b suffix on fwd a prefix (- +): a is reversed when b extends it to the left, b when its strand differs from a's.
__device__ __forceinline__ void gfa_link_fields(const u64 *edges, const uint16_t *len, u64 e, u32 &a, u32 &b, u32 &t, u32 &ov)
{
    u32 d, dt;
    edge_fields(edges, len, e, a, b, t, d, dt);
    ov = (u32)len[b - 1] - d;
}

__global__ void __launch_bounds__(256) gfa_link_len_kernel(const u64 *__restrict__ edges, const uint16_t *__restrict__ len, u64 e0, u64 n, u32 *__restrict__ out)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        u32 a, b, t, ov;
        gfa_link_fields(edges, len, e0 + i, a, b, t, ov);
        out[i] = (u32)(dec_digits(a) + dec_digits(b) + dec_digits(ov)) + 10u;
    }
}

__global__ void __launch_bounds__(256) gfa_link_fmt_kernel(const u64 *__restrict__ edges, const uint16_t *__restrict__ len, u64 e0, u64 n,
                                                            const u32 *__restrict__ off, char *__restrict__ out)
{
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        u32 a, b, t, ov;
        gfa_link_fields(edges, len, e0 + i, a, b, t, ov);
        char *p = out + off[i];
        *p++ = 'L'; *p++ = '\t'; p = put_dec(p, a); *p++ = '\t'; *p++ = t >= 2u ? '+' : '-'; *p++ = '\t';
        p = put_dec(p, b); *p++ = '\t'; *p++ = (t & 1u) ? '+' : '-'; *p++ = '\t';
        p = put_dec(p, ov); *p++ = 'M'; *p = '\n';
    }
}

static unsigned fmt_grid(u64 n)
{
    unsigned g = grid_for(n, 256, 2);
    return g > kSMs * 16u ? kSMs * 16u : g;
}

// lengths -> offsets -> text of one batch -> host buffer -> file
template <typename LenFn, typename FmtFn>
static bool write_batches(Context &c, FILE *f, u64 n_items, u64 per_batch, LenFn len_fn, FmtFn fmt_fn)
{
    cudaStream_t st = c.stream;
    std::vector<char> host;
    for (u64 i0 = 0; i0 < n_items; i0 += per_batch) {
        const u64 n = n_items - i0 < per_batch ? n_items - i0 : per_batch;
        ArenaScope arena_scope(c.arena, st);
        DevBuf<u32> lens(n, st), off(n, st), d_total(1, st);
        len_fn(i0, n, lens.p);
        exclusive_scan_u32(lens.p, off.p, n, d_total.p, st);
        u32 total = 0;
        SG_CUDA(cudaMemcpyAsync(&total, d_total.p, sizeof(u32), cudaMemcpyDeviceToHost, st));
        SG_CUDA(cudaStreamSynchronize(st));
        DevBuf<char> text(total, st);
        fmt_fn(i0, n, off.p, text.p);
        host.resize(total);
        SG_CUDA(cudaMemcpyAsync(host.data(), text.p, total, cudaMemcpyDeviceToHost, st));
        SG_CUDA(cudaStreamSynchronize(st));
        if (fwrite(host.data(), 1, total, f) != total) return false;
    }
    return true;
}

bool write_graph3_text(Context &c, FILE *f)
{
    cudaStream_t st = c.stream;
    // genomeSize (0 before step 5), numberOfReads, averageReadLength: overlapGraph.cpp:348-351
    fprintf(f, "0\n%llu\n%llu\n", (unsigned long long)c.cnt.good_reads, (unsigned long long)c.cnt.avg_len);
    const u64 E = c.cnt.n_edges;
    const u64 *edges = c.edges.p;
    const uint16_t *len = c.len.p;
    return write_batches(
        c, f, E, (u64)4 << 20,      // <= 78 bytes per edge: batches stay far below 2^32 bytes
        [&](u64 e0, u64 n, u32 *out) { edge_len_kernel<<<fmt_grid(n), 256, 0, st>>>(edges, len, e0, n, out); SG_LAUNCHED(); },
        [&](u64 e0, u64 n, const u32 *off, char *out) { edge_fmt_kernel<<<fmt_grid(n), 256, 0, st>>>(edges, len, e0, n, off, out); SG_LAUNCHED(); });
}

bool write_reads_text(Context &c, FILE *f)
{
    cudaStream_t st = c.stream;
    const u64 U = c.cnt.unique_reads;
    fprintf(f, "%llu\n", (unsigned long long)U);
    const u64 per_read = 2 * (u64)(c.max_len > 0 ? c.max_len : 1) + 16;
    u64 per_batch = ((u64)1 << 29) / per_read;            // <= 512 MB of text per batch
    if (per_batch < 1) per_batch = 1;
    const int SWS = c.SWS;
    return write_batches(
        c, f, U, per_batch,
        [&](u64 r0, u64 n, u32 *out) { read_len_kernel<<<fmt_grid(n), 256, 0, st>>>(c.len.p, c.freq.p, r0, n, out); SG_LAUNCHED(); },
        [&](u64 r0, u64 n, const u32 *off, char *out) {
            unsigned g = grid_for(n, 8, 1);
            if (g > kSMs * 16u) g = kSMs * 16u;
            read_fmt_kernel<<<g, 256, 0, st>>>(c.F.p, c.RC.p, c.len.p, c.freq.p, SWS, r0, n, off, out);
            SG_LAUNCHED();
        });
}

bool write_gfa_text(Context &c, FILE *f)
{
    cudaStream_t st = c.stream;
    if (fputs("H\tVN:Z:1.0\n", f) < 0) return false;
    // both kinds of line in batches of <= 256 MB of text: one host buffer of that size, offsets far below 2^32
    const u64 batch_bytes = (u64)1 << 28;
    const u64 U = c.cnt.unique_reads, E = c.cnt.n_edges;
    const u64 per_seg = (u64)(c.max_len > 0 ? c.max_len : 1) + 16 + 10 + 4 + 5;      // id, LN and RC values at their widest
    const u64 per_link = 10 + 10 + 10 + 4;                                            // two ids, an overlap of <= 4 digits
    const int SWS = c.SWS;
    const u64 *edges = c.edges.p;
    const uint16_t *len = c.len.p, *freq = c.freq.p;
    return write_batches(
               c, f, U, batch_bytes / per_seg,
               [&](u64 r0, u64 n, u32 *out) { gfa_seg_len_kernel<<<fmt_grid(n), 256, 0, st>>>(len, freq, r0, n, out); SG_LAUNCHED(); },
               [&](u64 r0, u64 n, const u32 *off, char *out) {
                   unsigned g = grid_for(n, 8, 1);
                   if (g > kSMs * 16u) g = kSMs * 16u;
                   gfa_seg_fmt_kernel<<<g, 256, 0, st>>>(c.F.p, len, freq, SWS, r0, n, off, out);
                   SG_LAUNCHED();
               }) &&
           write_batches(
               c, f, E, batch_bytes / per_link,
               [&](u64 e0, u64 n, u32 *out) { gfa_link_len_kernel<<<fmt_grid(n), 256, 0, st>>>(edges, len, e0, n, out); SG_LAUNCHED(); },
               [&](u64 e0, u64 n, const u32 *off, char *out) { gfa_link_fmt_kernel<<<fmt_grid(n), 256, 0, st>>>(edges, len, e0, n, off, out); SG_LAUNCHED(); });
}

}  // namespace sg
