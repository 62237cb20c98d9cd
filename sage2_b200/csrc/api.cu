// api.cu -- the C ABI of libsage2gpu (include/sage2gpu.h) over the stages in reads.cu, table.cu,
// search.cu and graph.cu, plus the host-side seams to the reference's formats.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "../../include/sage2gpu.h"
#include "context.h"

struct sage2gpu_ctx {
    sg::Context c;
};

namespace {

struct StageTimer {
    cudaEvent_t a, b;
    cudaStream_t st;
    explicit StageTimer(cudaStream_t s) : st(s)
    {
        cudaEventCreate(&a); cudaEventCreate(&b);
        cudaEventRecord(a, st);
    }
    float stop()
    {
        float ms = 0;
        cudaEventRecord(b, st);
        cudaEventSynchronize(b);
        cudaEventElapsedTime(&ms, a, b);
        return ms;
    }
    ~StageTimer() { cudaEventDestroy(a); cudaEventDestroy(b); }
};

template <typename Fn>
int guarded(sage2gpu_ctx *ctx, Fn fn)
{
    if (!ctx) return SAGE2GPU_ERR_ARG;
    try {
        SG_CUDA(cudaSetDevice(ctx->c.device));
        fn(ctx->c);
        if (ctx->c.opt_low_memory >= 2) {  // the stage's workspace goes back to the driver instead of waiting for the next stage
            SG_CUDA(cudaStreamSynchronize(ctx->c.stream));
            ctx->c.arena.destroy();
        }
        ctx->c.last_error.clear();
        return SAGE2GPU_OK;
    } catch (const sg::FormatError &e) {
        ctx->c.last_error = e.what();
        return SAGE2GPU_ERR_FORMAT;
    } catch (const sg::IoError &e) {
        ctx->c.last_error = e.what();
        return SAGE2GPU_ERR_IO;
    } catch (const sg::CudaError &e) {
        ctx->c.last_error = e.what();
        cudaGetLastError();
        return SAGE2GPU_ERR_CUDA;
    } catch (const std::exception &e) {
        ctx->c.last_error = e.what();
        return SAGE2GPU_ERR_STATE;
    }
}

void load_common(sg::Context &c, const uint8_t *bases, const int64_t *offsets, int64_t n, int k, bool dev, int rank = 0, int world = 1)
{
    SG_CHECK(k >= 1 && k < 65535, "min_overlap out of range");
    SG_CHECK(n == 0 || (bases != nullptr && offsets != nullptr), "null input");
    c.min_overlap = k;
    c.tm = sg::Timers();
    {
        StageTimer t(c.stream);
        sg::stage_ingest_ascii(c, bases, offsets, n, dev);
        c.tm.ingest = t.stop();
    }
    {
        StageTimer t(c.stream);
        sg::stage_organize_reads(c, rank, world);
        c.tm.sort_reads = t.stop();
    }
}

// record (word-big-endian) -> reference bytes (utils.cpp:96-119)
void record_to_bytes(const sg::u64 *rec, int len, uint8_t *out)
{
    const int nb = (len + 3) / 4;
    for (int b = 0; b < nb; ++b) out[b] = (uint8_t)(rec[b >> 3] >> (56 - 8 * (b & 7)));
}

struct HostReads {
    std::vector<uint16_t> len, freq;
    std::vector<sg::u64> F, RC;
};

void fetch_reads(sg::Context &c, HostReads &h)
{
    SG_CHECK(c.have_reads, "no reads loaded");
    const sg::u64 U = c.cnt.unique_reads;
    h.len.resize(U); h.freq.resize(U); h.F.resize(U * c.SWS); h.RC.resize(U * c.SWS);
    if (U == 0) return;
    SG_CUDA(cudaMemcpyAsync(h.len.data(), c.len.p, U * sizeof(uint16_t), cudaMemcpyDeviceToHost, c.stream));
    SG_CUDA(cudaMemcpyAsync(h.freq.data(), c.freq.p, U * sizeof(uint16_t), cudaMemcpyDeviceToHost, c.stream));
    SG_CUDA(cudaMemcpyAsync(h.F.data(), c.F.p, U * c.SWS * sizeof(sg::u64), cudaMemcpyDeviceToHost, c.stream));
    SG_CUDA(cudaMemcpyAsync(h.RC.data(), c.RC.p, U * c.SWS * sizeof(sg::u64), cudaMemcpyDeviceToHost, c.stream));
    SG_CUDA(cudaStreamSynchronize(c.stream));
}

void fetch_edges(sg::Context &c)
{
    SG_CHECK(c.have_graph, "overlap graph not built");
    const sg::u64 E = c.cnt.n_edges;
    if (c.h_edges.size() == 2 * E) return;
    c.h_edges.resize(2 * E);
    if (E) {
        SG_CUDA(cudaMemcpyAsync(c.h_edges.data(), c.edges.p, 2 * E * sizeof(sg::u64), cudaMemcpyDeviceToHost, c.stream));
        SG_CUDA(cudaStreamSynchronize(c.stream));
    }
}

}  // namespace

extern "C" {

int sage2gpu_create(sage2gpu_ctx **out, int device)
{
    if (!out) return SAGE2GPU_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return SAGE2GPU_ERR_CUDA;
    sage2gpu_ctx *ctx = new sage2gpu_ctx();
    ctx->c.device = device;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->c.stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return SAGE2GPU_ERR_CUDA;
    }
    // the search kernels gather random 32-byte sectors (slot index, partner reads): do not let L2 fetch
    // 64/128-byte granules from HBM for them
    cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, getenv("SAGE2GPU_L2_GRANULE") ? (size_t)atoi(getenv("SAGE2GPU_L2_GRANULE")) : 32);
    // keep freed blocks in the stream-ordered pool: steady-state allocation is a pointer bump
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    *out = ctx;
    return SAGE2GPU_OK;
}

void sage2gpu_destroy(sage2gpu_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->c.device);
    cudaStream_t st = ctx->c.stream;
    cudaStreamSynchronize(st);
    {
        sg::Context &c = ctx->c;
        c.d_bases.release(); c.d_offsets.release(); c.up_d_bases.release(); c.up_d_offsets.release(); c.up_d_freq.release(); c.raw.release(); c.F.release(); c.RC.release(); c.len.release(); c.freq.release();
        c.slots.release(); c.entries.release(); c.extR.release(); c.extL.release(); c.flag5.release();
        c.cont_max.release(); c.explored.release(); c.edges.release();
        sg::stage_mailbox_destroy(c);
        c.arena.destroy();
        c.pc_stage.release();
    }
    cudaStreamSynchronize(st);
    if (ctx->c.up_event) cudaEventDestroy(ctx->c.up_event);
    delete ctx;
    cudaStreamDestroy(st);
}

const char *sage2gpu_last_error(const sage2gpu_ctx *ctx) { return ctx ? ctx->c.last_error.c_str() : "null context"; }

int sage2gpu_load_reads(sage2gpu_ctx *ctx, const uint8_t *bases, const int64_t *offsets, int64_t n_reads, int min_overlap)
{
    return guarded(ctx, [&](sg::Context &c) { load_common(c, bases, offsets, n_reads, min_overlap, false); });
}

int sage2gpu_load_reads_device(sage2gpu_ctx *ctx, const uint8_t *d_bases, const int64_t *d_offsets, int64_t n_reads, int min_overlap)
{
    return guarded(ctx, [&](sg::Context &c) { load_common(c, d_bases, d_offsets, n_reads, min_overlap, true); });
}

// ---- several GPUs: the reads organised by key range, one range per rank (reads.cu) -----------------------------------
int sage2gpu_load_reads_partition(sage2gpu_ctx *ctx, const uint8_t *bases, const int64_t *offsets, int64_t n_reads, int min_overlap,
                                  int on_device, int rank, int world, uint64_t *unique_local)
{
    return guarded(ctx, [&](sg::Context &c) {
        load_common(c, bases, offsets, n_reads, min_overlap, on_device != 0, rank, world);
        if (unique_local) *unique_local = world > 1 ? c.rp_local : c.cnt.unique_reads;
    });
}

int sage2gpu_pack_slice(sage2gpu_ctx *ctx, const uint8_t *bases, const int64_t *offsets, int64_t n_reads, int min_overlap, int on_device,
                        int max_read_length, uint64_t *good_reads, uint64_t *total_bp, uint64_t *record_words)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(min_overlap >= 1 && min_overlap < 65535, "min_overlap out of range");
        SG_CHECK(max_read_length >= 1, "the longest read of the whole read set must be given");
        c.min_overlap = min_overlap;
        c.tm = sg::Timers();
        StageTimer t(c.stream);
        sg::stage_ingest_ascii(c, bases, offsets, n_reads, on_device != 0, max_read_length);
        c.tm.ingest = t.stop();
        if (good_reads) *good_reads = c.cnt.good_reads;
        if (total_bp) *total_bp = c.cnt.total_bp;
        if (record_words) *record_words = (uint64_t)c.SW;
    });
}

int sage2gpu_raw_gather_layout(sage2gpu_ctx *ctx, int rank, int world, const uint64_t *counts, void **records, uint64_t *first, uint64_t *total)
{
    return guarded(ctx, [&](sg::Context &c) {
        StageTimer t(c.stream);
        sg::u64 f = 0, tot = 0;
        sg::stage_raw_gather_layout(c, rank, world, (const sg::u64 *)counts, records, &f, &tot);
        if (first) *first = f;
        if (total) *total = tot;
        c.tm.ingest += t.stop();
    });
}

int sage2gpu_raw_gather_finish(sage2gpu_ctx *ctx, uint64_t total_reads, uint64_t good_reads, uint64_t total_bp)
{
    return guarded(ctx, [&](sg::Context &c) { sg::stage_raw_gather_finish(c, total_reads, good_reads, total_bp); });
}

int sage2gpu_organize_partition(sage2gpu_ctx *ctx, int rank, int world, uint64_t *unique_local)
{
    return guarded(ctx, [&](sg::Context &c) {
        StageTimer t(c.stream);
        sg::stage_organize_reads(c, rank, world);
        c.tm.sort_reads = t.stop();
        if (c.opt_low_memory) { SG_CUDA(cudaStreamSynchronize(c.stream)); c.arena.destroy(); }     // 25 GB of temporaries at 620 M reads
        if (unique_local) *unique_local = world > 1 ? c.rp_local : c.cnt.unique_reads;
    });
}

int sage2gpu_synth_reads(sage2gpu_ctx *ctx, uint8_t *d_bases, int64_t *d_offsets, uint64_t first_pair, uint64_t n_pairs, uint64_t genome_bp,
                         int read_length, float insert_mean, float insert_sd, uint64_t seed)
{
    return guarded(ctx, [&](sg::Context &c) { sg::stage_synth_reads(c, d_bases, d_offsets, first_pair, n_pairs, genome_bp, read_length, insert_mean, insert_sd, seed); });
}

// ---- helpers of a single-process multi-GPU host (host/sage2gpu_main.cpp --devices): no torch, no NCCL ---------------------
int sage2gpu_load_finish_packed(sage2gpu_ctx *ctx, uint64_t *n_reads, int *max_read_length, uint64_t *good_reads, uint64_t *total_bp)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.up_open, "sage2gpu_load_begin must be called first");
        c.up_open = false;
        SG_CUDA(cudaEventSynchronize(c.up_event));
        StageTimer t(c.stream);
        // pass 1 finds the longest read, pass 2 packs with that stride into the slice buffer (the joint array comes later)
        sg::stage_ingest_ascii(c, c.up_d_bases.p, c.up_d_offsets.p, (int64_t)c.up_reads, true, -1);
        c.up_d_bases.release(); c.up_d_offsets.release();
        c.tm.ingest = t.stop();
        if (n_reads) *n_reads = c.n_input;
        if (max_read_length) *max_read_length = c.max_len;
        if (good_reads) *good_reads = c.cnt.good_reads;
        if (total_bp) *total_bp = c.cnt.total_bp;
    });
}

int sage2gpu_load_max_length(sage2gpu_ctx *ctx, int *max_read_length)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.up_open, "sage2gpu_load_begin must be called first");
        SG_CHECK(max_read_length != nullptr, "null argument");
        SG_CUDA(cudaEventSynchronize(c.up_event));
        *max_read_length = sg::stage_uploaded_max_len(c);
    });
}

int sage2gpu_load_finish_slice(sage2gpu_ctx *ctx, int max_read_length, uint64_t *n_reads, uint64_t *good_reads, uint64_t *total_bp,
                               uint64_t *record_words)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.up_open, "sage2gpu_load_begin must be called first");
        SG_CHECK(max_read_length >= 1, "the longest read of the whole read set must be given");
        c.up_open = false;
        SG_CUDA(cudaEventSynchronize(c.up_event));
        StageTimer t(c.stream);
        sg::stage_ingest_ascii(c, c.up_d_bases.p, c.up_d_offsets.p, (int64_t)c.up_reads, true, max_read_length);
        c.up_d_bases.release(); c.up_d_offsets.release();
        c.tm.ingest = t.stop();
        if (n_reads) *n_reads = c.n_input;
        if (good_reads) *good_reads = c.cnt.good_reads;
        if (total_bp) *total_bp = c.cnt.total_bp;
        if (record_words) *record_words = (uint64_t)c.SW;
    });
}

int sage2gpu_table_bytes(sage2gpu_ctx *ctx, int world, uint64_t *replicated_slot_bytes, uint64_t *replicated_entry_bytes,
                         uint64_t *sharded_slot_bytes, uint64_t *sharded_entry_bytes, uint64_t *device_free_bytes)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.have_reads, "the reads must be organised first");
        SG_CHECK(world >= 1 && world <= sg::kMaxWorld, "bad world");
        const sg::u64 U = c.cnt.unique_reads;
        // stage_build_table: no table for an empty read set; at most 4U entries (one per key of a bucket), in any shard
        const sg::u64 shard = U ? sg::table_shard_slots(U, world) * sizeof(sg::u64) : 0, entries = 4 * U * sizeof(sg::u32);
        if (replicated_slot_bytes) *replicated_slot_bytes = shard * (sg::u64)world;
        if (replicated_entry_bytes) *replicated_entry_bytes = entries;
        if (sharded_slot_bytes) *sharded_slot_bytes = shard;
        if (sharded_entry_bytes) *sharded_entry_bytes = entries;
        if (device_free_bytes) {
            size_t fr = 0, tot = 0;
            SG_CUDA(cudaStreamSynchronize(c.stream));
            SG_CUDA(cudaMemGetInfo(&fr, &tot));
            *device_free_bytes = fr;
        }
    });
}

int sage2gpu_peer_copy(sage2gpu_ctx *dst, void *dst_ptr, sage2gpu_ctx *src, const void *src_ptr, uint64_t n_bytes)
{
    if (!dst || !src) return SAGE2GPU_ERR_ARG;
    return guarded(dst, [&](sg::Context &c) {
        if (n_bytes == 0) return;
        SG_CHECK(dst_ptr && src_ptr, "null pointer");
        // both contexts' streams are idle between the stages of the host's schedule; a synchronous peer copy keeps it simple
        SG_CUDA(cudaMemcpyPeer(dst_ptr, c.device, src_ptr, src->c.device, (size_t)n_bytes));
    });
}

int sage2gpu_phase_a_import(sage2gpu_ctx *ctx, sage2gpu_ctx *src, int src_rank)
{
    if (!ctx || !src) return SAGE2GPU_ERR_ARG;
    return guarded(ctx, [&](sg::Context &c) { sg::stage_phase_a_import(c, src->c, src_rank); });
}

int sage2gpu_reads_gather_layout(sage2gpu_ctx *ctx, const uint64_t *counts, void **records, void **lengths, void **frequencies,
                                 uint64_t *first, uint64_t *total, uint64_t *record_stride_words)
{
    return guarded(ctx, [&](sg::Context &c) {
        StageTimer t(c.stream);
        sg::u64 f = 0, tot = 0;
        sg::stage_reads_gather_layout(c, (const sg::u64 *)counts, records, lengths, frequencies, &f, &tot);
        if (first) *first = f;
        if (total) *total = tot;
        if (record_stride_words) *record_stride_words = (uint64_t)c.SWS;
        c.tm.sort_reads += t.stop();
    });
}

int sage2gpu_reads_gather_finish(sage2gpu_ctx *ctx)
{
    return guarded(ctx, [&](sg::Context &c) {
        StageTimer t(c.stream);
        sg::stage_reads_gather_finish(c);
        c.tm.sort_reads += t.stop();
    });
}

// ---- several GPUs, replicated table: one key-hash shard built per rank, the shards all-gathered (table.cu) --------------
int sage2gpu_build_hash_table_part(sage2gpu_ctx *ctx, int rank, int world)
{
    return guarded(ctx, [&](sg::Context &c) {
        StageTimer t(c.stream);
        sg::stage_build_table(c, rank, world, true);
        c.tm.build_table = t.stop();
    });
}

int sage2gpu_table_shard_info(sage2gpu_ctx *ctx, uint64_t *slots, uint64_t *entries, uint64_t *distinct_keys, uint64_t *keys_over_threshold)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.have_table, "no table built");
        if (slots) *slots = c.cap;
        if (entries) *entries = c.tb_entries;
        if (distinct_keys) *distinct_keys = c.cnt.distinct_keys;
        if (keys_over_threshold) *keys_over_threshold = c.cnt.keys_over_threshold;
    });
}

int sage2gpu_table_gather_layout(sage2gpu_ctx *ctx, const uint64_t *entry_counts, void **slots, void **entries, uint64_t *slots_per_shard,
                                 uint64_t *entries_first)
{
    return guarded(ctx, [&](sg::Context &c) {
        StageTimer t(c.stream);
        sg::u64 sps = 0, ef = 0;
        sg::stage_table_gather_layout(c, (const sg::u64 *)entry_counts, slots, entries, &sps, &ef);
        if (slots_per_shard) *slots_per_shard = sps;
        if (entries_first) *entries_first = ef;
        c.tm.build_table += t.stop();
    });
}

int sage2gpu_table_gather_finish(sage2gpu_ctx *ctx, const uint64_t *entry_counts, const uint64_t *distinct_keys, const uint64_t *keys_over_threshold)
{
    return guarded(ctx, [&](sg::Context &c) {
        StageTimer t(c.stream);
        sg::stage_table_gather_finish(c, (const sg::u64 *)entry_counts, (const sg::u64 *)distinct_keys, (const sg::u64 *)keys_over_threshold);
        c.tm.build_table += t.stop();
    });
}

// ---- streamed upload: the FASTA/Q parser fills one pinned chunk while the previous one is copied ----
int sage2gpu_load_begin(sage2gpu_ctx *ctx, int min_overlap)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(min_overlap >= 1 && min_overlap < 65535, "min_overlap out of range");
        c.min_overlap = min_overlap;
        c.tm = sg::Timers();
        c.have_reads = c.have_table = c.have_graph = false;
        c.up_reads = 0; c.up_bases = 0; c.up_open = true;
        if (!c.up_event) SG_CUDA(cudaEventCreateWithFlags(&c.up_event, cudaEventDisableTiming));
    });
}

int sage2gpu_load_append(sage2gpu_ctx *ctx, const uint8_t *bases, const int64_t *offsets, int64_t n_reads)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.up_open, "sage2gpu_load_begin must be called first");
        SG_CHECK(n_reads >= 0 && (n_reads == 0 || (bases && offsets)), "bad chunk");
        SG_CUDA(cudaEventSynchronize(c.up_event));          // the previous chunk's host buffers are free again
        if (n_reads == 0) return;
        sg::stage_upload_chunk(c, bases, offsets, n_reads);
        SG_CUDA(cudaEventRecord(c.up_event, c.stream));
    });
}

int sage2gpu_load_append_text(sage2gpu_ctx *ctx, const uint8_t *text, uint64_t n_bytes, int is_final, int *marker,
                              uint64_t max_records, uint64_t *consumed, uint64_t *n_records)
{
    bool regular = true;
    int rc = guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.up_open, "sage2gpu_load_begin must be called first");
        SG_CHECK(marker && consumed && n_records && (n_bytes == 0 || text), "null argument");
        SG_CUDA(cudaEventSynchronize(c.up_event));
        sg::u64 used = 0, nrec = 0;
        regular = sg::stage_parse_text_chunk(c, text, n_bytes, is_final != 0, *marker, max_records, used, nrec);
        *consumed = used; *n_records = nrec;
    });
    if (rc == 0 && !regular) { ctx->c.last_error = "text is not in the regular 4-line FASTQ / 2-line FASTA layout"; return SAGE2GPU_ERR_FORMAT; }
    return rc;
}

int sage2gpu_load_count(sage2gpu_ctx *ctx, uint64_t *n_reads)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.up_open && n_reads, "sage2gpu_load_begin must be called first");
        *n_reads = c.up_reads;
    });
}

int sage2gpu_load_remove(sage2gpu_ctx *ctx, uint64_t first, uint64_t count)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.up_open, "sage2gpu_load_begin must be called first");
        SG_CUDA(cudaEventSynchronize(c.up_event));
        sg::stage_remove_uploaded(c, first, count);
    });
}

int sage2gpu_load_finish(sage2gpu_ctx *ctx)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.up_open, "sage2gpu_load_begin must be called first");
        c.up_open = false;
        SG_CUDA(cudaEventSynchronize(c.up_event));
        {
            StageTimer t(c.stream);
            sg::stage_ingest_ascii(c, c.up_d_bases.p, c.up_d_offsets.p, (int64_t)c.up_reads, true);
            c.up_d_bases.release(); c.up_d_offsets.release();
            c.tm.ingest = t.stop();
        }
        {
            StageTimer t(c.stream);
            sg::stage_organize_reads(c);
            c.tm.sort_reads = t.stop();
        }
    });
}

// ---- a saved .reads file (ReadLoader::loadReadsFromFile, readLoader.cpp:289): parse.cu, reads.cu ----------------------------
int sage2gpu_saved_reads_info(sage2gpu_ctx *ctx, const char *path, uint64_t *n_reads, uint64_t *body_bytes)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(path != nullptr, "null path");
        sg::u64 u = 0, off = 0, body = 0;
        sg::saved_reads_header(path, u, off, body);
        if (n_reads) *n_reads = u;
        if (body_bytes) *body_bytes = body;
    });
}

int sage2gpu_saved_reads_slice(sage2gpu_ctx *ctx, const char *path, int min_overlap, uint64_t byte_begin, uint64_t byte_end, uint64_t *n_lines,
                               int *max_read_length, uint64_t *bad_line)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(path != nullptr, "null path");
        SG_CHECK(min_overlap >= 1 && min_overlap < 65535, "min_overlap out of range");
        if (bad_line) *bad_line = 0;
        c.min_overlap = min_overlap;
        c.tm = sg::Timers();
        c.up_open = false;
        c.have_reads = c.have_table = c.have_graph = false;
        StageTimer t(c.stream);
        sg::u64 n = 0;
        int ml = 0;
        try {
            sg::stage_parse_saved_reads(c, path, byte_begin, byte_end, n, ml);
        } catch (const sg::FormatError &e) {
            if (bad_line) *bad_line = e.line;
            c.up_reads = c.up_bases = 0;
            c.up_d_bases.release(); c.up_d_offsets.release(); c.up_d_freq.release();
            throw;
        }
        c.tm.ingest = t.stop();
        if (n_lines) *n_lines = n;
        if (max_read_length) *max_read_length = ml;
    });
}

int sage2gpu_saved_reads_pack(sage2gpu_ctx *ctx, int rank, int world, int max_read_length, uint64_t *unique_local, uint64_t *good_reads,
                              uint64_t *total_bp)
{
    return guarded(ctx, [&](sg::Context &c) {
        const sg::u64 good = c.sr_good, bp = c.sr_bp;
        StageTimer t(c.stream);
        sg::stage_pack_saved_reads(c, rank, world, max_read_length);
        c.tm.sort_reads = t.stop();
        if (c.opt_low_memory) { SG_CUDA(cudaStreamSynchronize(c.stream)); c.arena.destroy(); }
        if (unique_local) *unique_local = c.rp_local;
        if (good_reads) *good_reads = good;
        if (total_bp) *total_bp = bp;
    });
}

int sage2gpu_saved_reads_finish(sage2gpu_ctx *ctx, uint64_t n_reads, uint64_t good_reads, uint64_t total_bp, uint64_t *bad_line)
{
    return guarded(ctx, [&](sg::Context &c) {
        if (bad_line) *bad_line = 0;
        StageTimer t(c.stream);
        try {
            sg::stage_check_saved_reads(c, n_reads, good_reads, total_bp);
        } catch (const sg::FormatError &e) {
            if (bad_line) *bad_line = e.line;
            throw;
        }
        c.tm.sort_reads += t.stop();
    });
}

int sage2gpu_load_saved_reads(sage2gpu_ctx *ctx, const char *path, int min_overlap)
{
    // the one-slice case of the calls above; a line of the slice is line + 1 of the file (line 1 is the number of reads)
    uint64_t U = 0, body = 0, n = 0, good = 0, bp = 0, bad = 0;
    int ml = 0;
    int rc = sage2gpu_saved_reads_info(ctx, path, &U, &body);
    if (rc == 0) {
        rc = sage2gpu_saved_reads_slice(ctx, path, min_overlap, 0, body, &n, &ml, &bad);
        if (rc == SAGE2GPU_ERR_FORMAT) {
            const std::string m = ctx->c.last_error;
            ctx->c.last_error = "line " + std::to_string(bad + 1) + m.substr(m.find(':'));
        }
    }
    if (rc == 0) rc = sage2gpu_saved_reads_pack(ctx, 0, 1, ml, nullptr, &good, &bp);
    if (rc == 0) rc = sage2gpu_saved_reads_finish(ctx, U, good, bp, nullptr);
    return rc;
}

void *sage2gpu_host_alloc(uint64_t n_bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, n_bytes ? n_bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

void sage2gpu_host_free(void *p) { if (p) cudaFreeHost(p); }

int sage2gpu_build_hash_table(sage2gpu_ctx *ctx)
{
    return guarded(ctx, [&](sg::Context &c) {
        StageTimer t(c.stream);
        sg::stage_build_table(c);
        c.tm.build_table = t.stop();
    });
}

static void finish_graph(sg::Context &c)
{
    SG_CHECK(c.have_phase_a, "phase A must run first");
    if (!c.have_phase_b) {      // (a sharded build ran it already: the reads left for phase C had to be routed first)
        StageTimer t(c.stream);
        sg::stage_phase_b(c);
        c.tm.phase_b = t.stop();
    }
    sg::stage_phase_c_and_finalize(c);
    c.have_phase_b = false;
    c.tm.total_device = c.tm.ingest + c.tm.sort_reads + c.tm.build_table + c.tm.phase_a + c.tm.phase_b +
                        c.tm.phase_c_dev + c.tm.phase_c_host + c.tm.sort_edges;
}

int sage2gpu_phase_a_partition(sage2gpu_ctx *ctx, int rank, int world)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.have_table, "build_hash_table must run first");
        StageTimer t(c.stream);
        sg::stage_phase_a(c, rank, world);
        c.tm.phase_a = t.stop();
    });
}

int sage2gpu_phase_a_buffers(sage2gpu_ctx *ctx, void **right_ext, void **left_ext, void **over_limit, void **contained_by,
                             uint64_t *reads_per_rank, uint64_t *unique_reads)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.have_phase_a, "phase A must run first");
        if (right_ext) *right_ext = c.extR.p;
        if (left_ext) *left_ext = c.extL.p;
        if (over_limit) *over_limit = c.flag5.p;
        if (contained_by) *contained_by = c.cont_max.p;
        if (reads_per_rank) *reads_per_rank = c.pa_chunk;
        if (unique_reads) *unique_reads = c.cnt.unique_reads;
    });
}

int sage2gpu_table_view(sage2gpu_ctx *ctx, const void **slots, uint64_t *n_slots, const void **entries, uint64_t *n_entries,
                        uint64_t *sectors_per_shard, uint64_t *shards)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.have_table, "no table built");
        SG_CHECK(!c.tb_joint || c.tb_shards > 1, "sage2gpu_table_gather_finish must run first");
        if (slots) *slots = c.slots.p;
        if (n_slots) *n_slots = c.cap;
        if (entries) *entries = c.entries.p;
        if (n_entries) *n_entries = c.tb_entries;
        if (sectors_per_shard) *sectors_per_shard = c.cap / sg::kSlotsPerSector / (sg::u64)c.tb_shards;
        if (shards) *shards = (uint64_t)c.tb_shards;
    });
}

int sage2gpu_finish_graph(sage2gpu_ctx *ctx)
{
    return guarded(ctx, [&](sg::Context &c) { finish_graph(c); });
}

// ---- sharded table (SURVEY 8(e)) -----------------------------------------------------------------------------------
int sage2gpu_build_hash_table_shard(sage2gpu_ctx *ctx, int rank, int world)
{
    return guarded(ctx, [&](sg::Context &c) {
        StageTimer t(c.stream);
        sg::stage_build_table(c, rank, world);
        c.tm.build_table = t.stop();
    });
}

int sage2gpu_phase_a_sharded_begin(sage2gpu_ctx *ctx, int rank, int world, uint64_t *first, uint64_t *count)
{
    return guarded(ctx, [&](sg::Context &c) {
        sg::stage_phase_a_sharded_begin(c, rank, world);
        c.tm.phase_a = 0;
        if (first) *first = c.pa_lo;
        if (count) *count = c.pa_hi - c.pa_lo;
    });
}

int sage2gpu_route_begin(sage2gpu_ctx *ctx, int what, uint64_t first, uint64_t count, int exact, int world, void **queries,
                         uint64_t *counts, uint64_t *n_reads)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(counts != nullptr, "null counts");
        StageTimer t(c.stream);
        sg::stage_route_begin(c, what, first, count, exact, world, queries, counts);
        if (n_reads) *n_reads = c.rt_n;
        (what == 1 ? c.tm.phase_c_dev : c.tm.phase_a) += t.stop();
    });
}

int sage2gpu_shard_answer(sage2gpu_ctx *ctx, const void *queries, const uint64_t *counts_per_source, int exact, int world, void **responses,
                          void **entries, uint64_t *entry_counts)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(counts_per_source && responses && entries && entry_counts, "null argument");
        StageTimer t(c.stream);
        sg::stage_shard_answer(c, queries, counts_per_source, exact, world, responses, entries, entry_counts);
        c.tm.phase_a += t.stop();
    });
}

int sage2gpu_route_finish(sage2gpu_ctx *ctx, const void *responses, const void *entries, const uint64_t *entry_counts)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(entry_counts != nullptr, "null entry counts");
        StageTimer t(c.stream);
        sg::stage_route_finish(c, responses, entries, entry_counts);
        (c.rt_what == 1 ? c.tm.phase_c_dev : c.tm.phase_a) += t.stop();
    });
}

int sage2gpu_mailbox_create(sage2gpu_ctx *ctx, int rank, int world, uint64_t max_reads_per_batch, void *ipc_handle_out, void **local_ptr)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.have_reads, "load the reads first: the mailbox is sized for their window count");
        const int wstride = c.max_len - c.h + 1 > 1 ? c.max_len - c.h + 1 : 1;
        sg::stage_mailbox_create(c, rank, world, (max_reads_per_batch ? max_reads_per_batch : 1) * (sg::u64)wstride, ipc_handle_out, local_ptr);
    });
}

int sage2gpu_mailbox_open(sage2gpu_ctx *ctx, int peer_rank, const void *ipc_handle, void *ptr)
{
    return guarded(ctx, [&](sg::Context &c) { sg::stage_mailbox_open(c, peer_rank, ipc_handle, ptr); });
}

int sage2gpu_mailbox_barrier(sage2gpu_ctx *ctx)
{
    return guarded(ctx, [&](sg::Context &c) { sg::stage_mailbox_barrier(c); });
}

int sage2gpu_route_post(sage2gpu_ctx *ctx, int what, uint64_t first, uint64_t count, int exact, uint64_t *n_reads, uint64_t *bytes_sent)
{
    return guarded(ctx, [&](sg::Context &c) {
        StageTimer t(c.stream);
        sg::stage_route_post(c, what, first, count, exact, n_reads);
        if (bytes_sent) {
            *bytes_sent = 0;
            for (int g = 0; g < c.mb.world; ++g) if (g != c.mb.rank) *bytes_sent += c.rt_counts[g] * (exact ? 16 : 8);
        }
        (what == 1 ? c.tm.phase_c_dev : c.tm.phase_a) += t.stop();
    });
}

int sage2gpu_answer_post(sage2gpu_ctx *ctx, int exact, uint64_t *bytes_sent)
{
    return guarded(ctx, [&](sg::Context &c) {
        StageTimer t(c.stream);
        sg::stage_answer_post(c, exact, bytes_sent);
        c.tm.phase_a += t.stop();
    });
}

int sage2gpu_route_collect(sage2gpu_ctx *ctx)
{
    return guarded(ctx, [&](sg::Context &c) {
        StageTimer t(c.stream);
        sg::stage_route_collect(c);
        (c.rt_what == 1 ? c.tm.phase_c_dev : c.tm.phase_a) += t.stop();
    });
}

int sage2gpu_phase_a_routed(sage2gpu_ctx *ctx, uint64_t *n_redo)
{
    return guarded(ctx, [&](sg::Context &c) {
        StageTimer t(c.stream);
        const sg::u64 r = sg::stage_phase_a_routed(c);
        if (n_redo) *n_redo = r;
        c.tm.phase_a += t.stop();
    });
}

int sage2gpu_phase_a_sharded_end(sage2gpu_ctx *ctx)
{
    return guarded(ctx, [&](sg::Context &c) { sg::stage_phase_a_sharded_end(c); });
}

int sage2gpu_map_reads(sage2gpu_ctx *ctx, const uint8_t *bases, const int64_t *offsets, int64_t n_reads, int on_device, int64_t *ids,
                       uint8_t *good, float *kernel_ms)
{
    return guarded(ctx, [&](sg::Context &c) {
        const float ms = sg::stage_map_reads(c, bases, offsets, n_reads, on_device != 0, ids, good);
        if (kernel_ms) *kernel_ms = ms;
    });
}

int sage2gpu_phase_b(sage2gpu_ctx *ctx)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.have_phase_a, "phase A must run first");
        StageTimer t(c.stream);
        sg::stage_phase_b(c);
        c.tm.phase_b = t.stop();
    });
}

int sage2gpu_build_overlap_graph(sage2gpu_ctx *ctx)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.have_table, "build_hash_table must run first");
        {
            StageTimer t(c.stream);
            sg::stage_phase_a(c);
            c.tm.phase_a = t.stop();
        }
        finish_graph(c);
    });
}

int sage2gpu_run_steps123(sage2gpu_ctx *ctx, const uint8_t *bases, const int64_t *offsets, int64_t n_reads, int min_overlap)
{
    int rc = sage2gpu_load_reads(ctx, bases, offsets, n_reads, min_overlap);
    if (rc) return rc;
    rc = sage2gpu_build_hash_table(ctx);
    if (rc) return rc;
    return sage2gpu_build_overlap_graph(ctx);
}

int sage2gpu_get_counters(const sage2gpu_ctx *ctx, sage2gpu_counters *o)
{
    if (!ctx || !o) return SAGE2GPU_ERR_ARG;
    const sg::Counters &n = ctx->c.cnt;
    o->total_reads = n.total_reads; o->good_reads = n.good_reads; o->unique_reads = n.unique_reads;
    o->total_bp = n.total_bp; o->avg_len = n.avg_len;
    o->hash_len = n.hash_len; o->distinct_keys = n.distinct_keys; o->keys_over_threshold = n.keys_over_threshold;
    o->table_capacity = n.table_capacity;
    o->contained_ext = n.contained_ext; o->contained_size = n.contained_size; o->left_to_explore = n.left_to_explore;
    o->edges_phase_b = n.edges_phase_b; o->candidates_c = n.candidates_c; o->edges_inserted_c = n.edges_inserted_c;
    o->transitive_removed = n.transitive_removed; o->n_edges = n.n_edges;
    o->compare_calls = n.compare_calls; o->window_probes = n.window_probes; o->slow_path_reads = n.slow_path_reads;
    o->record_words = (uint64_t)ctx->c.SW;
    o->probe_restarts = n.probe_restarts;
    o->phase_c_on_device = n.phase_c_on_device;
    o->fast_path_reads = n.fast_path_reads;
    return SAGE2GPU_OK;
}

int sage2gpu_get_timers(const sage2gpu_ctx *ctx, sage2gpu_timers *o)
{
    if (!ctx || !o) return SAGE2GPU_ERR_ARG;
    const sg::Timers &t = ctx->c.tm;
    o->ingest = t.ingest; o->sort_reads = t.sort_reads; o->build_table = t.build_table; o->phase_a = t.phase_a;
    o->phase_b = t.phase_b; o->phase_c_dev = t.phase_c_dev; o->phase_c_host = t.phase_c_host;
    o->sort_edges = t.sort_edges; o->total = t.total_device; o->phase_a_kernel = t.phase_a_kernel;
    return SAGE2GPU_OK;
}

void *sage2gpu_stream(const sage2gpu_ctx *ctx) { return ctx ? (void *)ctx->c.stream : nullptr; }

int sage2gpu_reads_bytes(const sage2gpu_ctx *ctx, uint64_t *n_bytes)
{
    if (!ctx || !n_bytes) return SAGE2GPU_ERR_ARG;
    sage2gpu_ctx *m = const_cast<sage2gpu_ctx *>(ctx);
    return guarded(m, [&](sg::Context &c) {
        SG_CHECK(c.have_reads, "no reads loaded");
        const sg::u64 U = c.cnt.unique_reads;
        std::vector<uint16_t> len(U);
        if (U) {
            SG_CUDA(cudaMemcpyAsync(len.data(), c.len.p, U * sizeof(uint16_t), cudaMemcpyDeviceToHost, c.stream));
            SG_CUDA(cudaStreamSynchronize(c.stream));
        }
        uint64_t tot = 0;
        for (sg::u64 i = 0; i < U; ++i) tot += (uint64_t)(len[i] + 3) / 4;
        *n_bytes = tot;
    });
}

int sage2gpu_get_reads(sage2gpu_ctx *ctx, uint16_t *length, uint16_t *frequency, uint64_t *byte_off, uint8_t *fwd, uint8_t *rc)
{
    return guarded(ctx, [&](sg::Context &c) {
        HostReads h;
        fetch_reads(c, h);
        const sg::u64 U = c.cnt.unique_reads;
        uint64_t off = 0;
        for (sg::u64 i = 0; i < U; ++i) {
            if (length) length[i] = h.len[i];
            if (frequency) frequency[i] = h.freq[i];
            if (byte_off) byte_off[i] = off;
            if (fwd) record_to_bytes(&h.F[i * c.SWS], h.len[i], fwd + off);
            if (rc) record_to_bytes(&h.RC[i * c.SWS], h.len[i], rc + off);
            off += (uint64_t)(h.len[i] + 3) / 4;
        }
        if (byte_off) byte_off[U] = off;
    });
}

int sage2gpu_get_extensions(sage2gpu_ctx *ctx, uint64_t *right_ext, uint64_t *left_ext, uint8_t *explored)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.have_graph, "overlap graph not built");
        const sg::u64 U = c.cnt.unique_reads;
        if (U == 0) return;
        if (right_ext) SG_CUDA(cudaMemcpyAsync(right_ext, c.extR.p, U * sizeof(uint64_t), cudaMemcpyDeviceToHost, c.stream));
        if (left_ext) SG_CUDA(cudaMemcpyAsync(left_ext, c.extL.p, U * sizeof(uint64_t), cudaMemcpyDeviceToHost, c.stream));
        if (explored) SG_CUDA(cudaMemcpyAsync(explored, c.explored.p, U, cudaMemcpyDeviceToHost, c.stream));
        SG_CUDA(cudaStreamSynchronize(c.stream));
    });
}

int sage2gpu_get_edges(sage2gpu_ctx *ctx, sage2gpu_edge *out, uint64_t capacity, uint64_t *n_edges)
{
    return guarded(ctx, [&](sg::Context &c) {
        fetch_edges(c);
        const sg::u64 E = c.cnt.n_edges;
        if (n_edges) *n_edges = E;
        if (!out) return;
        SG_CHECK(capacity >= E, "edge buffer too small");
        std::vector<uint16_t> len(c.cnt.unique_reads);
        if (!len.empty()) {
            SG_CUDA(cudaMemcpyAsync(len.data(), c.len.p, len.size() * sizeof(uint16_t), cudaMemcpyDeviceToHost, c.stream));
            SG_CUDA(cudaStreamSynchronize(c.stream));
        }
        for (sg::u64 e = 0; e < E; ++e) {
            const sg::u64 w0 = c.h_edges[2 * e], w1 = c.h_edges[2 * e + 1];
            sage2gpu_edge &x = out[e];
            x.from = w0 >> 32; x.to = w0 & 0xFFFFFFFFull;
            x.type = (uint32_t)(w1 >> 20) & 3u; x.delta = (uint32_t)(w1 & 0xFFFFFu);
            const uint32_t ul = len[x.from - 1], vl = len[x.to - 1];
            x.delta_twin = ul - (vl - x.delta);                    // overlapGraph.cpp:147
            x.reserved = 0;
        }
    });
}

int sage2gpu_get_edges_packed(sage2gpu_ctx *ctx, uint64_t *out, uint64_t capacity, uint64_t *n_edges)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.have_graph, "overlap graph not built");
        const sg::u64 E = c.cnt.n_edges;
        if (n_edges) *n_edges = E;
        if (!out || E == 0) return;
        SG_CHECK(capacity >= E, "edge buffer too small");
        SG_CUDA(cudaMemcpyAsync(out, c.edges.p, 2 * E * sizeof(sg::u64), cudaMemcpyDeviceToHost, c.stream));
        SG_CUDA(cudaStreamSynchronize(c.stream));
    });
}

int sage2gpu_measure_gather(sage2gpu_ctx *ctx, uint64_t footprint_bytes, int granule_bytes, uint64_t n_loads, int mode, double *gbps)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(gbps != nullptr, "null result pointer");
        sg::ArenaScope arena_scope(c.arena, c.stream);
        *gbps = (double)sg::gather_bench(footprint_bytes, granule_bytes, n_loads, mode, c.stream);
    });
}

int sage2gpu_digest(sage2gpu_ctx *ctx, uint64_t *reads_digest, uint64_t *edges_digest)
{
    return guarded(ctx, [&](sg::Context &c) {
        sg::u64 r = 0, e = 0;
        sg::stage_digest(c, reads_digest ? &r : nullptr, edges_digest ? &e : nullptr);
        if (reads_digest) *reads_digest = r;
        if (edges_digest) *edges_digest = e;
    });
}

int sage2gpu_set_option(sage2gpu_ctx *ctx, const char *name, int64_t value)
{
    return guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(name != nullptr, "null option name");
        const std::string n(name);
        if (n == "read_order") { SG_CHECK(value >= -1 && value <= 1, "read_order: -1 default, 0 id order, 1 min-hash order"); c.opt_read_order = (int)value; }
        else if (n == "low_memory") {
            SG_CHECK(value >= 0 && value <= 2, "low_memory: 0, 1 or 2");
            c.opt_low_memory = (int)value; c.arena.tight = value > 0;
            if (value > 0 && c.have_reads) {
                // switched on after the reads were organised: release now what the mode would have released by then -- the packed
                // input, this context's packed slice and its unique run before the gather -- and the workspace
                SG_CUDA(cudaStreamSynchronize(c.stream));
                c.raw.release(); c.raw_slice.release(); c.F_loc.release(); c.len_loc.release(); c.freq_loc.release();
                c.arena.destroy();
                sg::trim_default_pool(c.device, c.stream);
            }
        }
        else if (n == "fast_scan") { SG_CHECK(value >= -1 && value <= 1, "fast_scan: -1 default, 0 off, 1 on"); c.opt_fast_scan = (int)value; }
        else throw sg::CudaError("unknown option: " + n);
    });
}

uint64_t sage2gpu_kernel_launches(void) { return sg::launch_counter(); }

int sage2gpu_write_reads(sage2gpu_ctx *ctx, const char *path)
{
    int io = 0;
    int rc = guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.have_reads, "no reads loaded");
        FILE *f = fopen(path, "wb");
        if (!f) { io = 1; return; }
        bool ok = false;
        try { ok = sg::write_reads_text(c, f); } catch (...) { fclose(f); throw; }
        if (fclose(f) != 0 || !ok) io = 1;
    });
    if (rc == 0 && io) { ctx->c.last_error = std::string("cannot write ") + path; return SAGE2GPU_ERR_IO; }
    return rc;
}

int sage2gpu_write_graph3(sage2gpu_ctx *ctx, const char *path)
{
    int io = 0;
    int rc = guarded(ctx, [&](sg::Context &c) {
        SG_CHECK(c.have_graph, "overlap graph not built");
        FILE *f = fopen(path, "wb");
        if (!f) { io = 1; return; }
        bool ok = false;
        try { ok = sg::write_graph3_text(c, f); } catch (...) { fclose(f); throw; }
        if (fclose(f) != 0 || !ok) io = 1;
    });
    if (rc == 0 && io) { ctx->c.last_error = std::string("cannot write ") + path; return SAGE2GPU_ERR_IO; }
    return rc;
}

}  // extern "C"
