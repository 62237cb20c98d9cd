// context.h -- device-resident state of one libsage2gpu context (one GPU, one stream).
#pragma once
#include <stdio.h>
#include <string>
#include <vector>
#include "core.cuh"
#include "device_utils.cuh"

namespace sg {

struct Counters {
    // step 1 (readLoader.cpp:164-169,257)
    u64 total_reads = 0, good_reads = 0, unique_reads = 0, total_bp = 0, avg_len = 0;
    // step 2 (hashTable.cpp:86,124)
    u64 hash_len = 0, distinct_keys = 0, keys_over_threshold = 0, table_capacity = 0;
    // step 3 (economyGraph.cpp:485-487,569-571)
    u64 contained_ext = 0, contained_size = 0, left_to_explore = 0;
    u64 edges_phase_b = 0, candidates_c = 0, edges_inserted_c = 0, transitive_removed = 0;
    u64 n_edges = 0;
    u64 compare_calls = 0;   // V of SURVEY 8(d) (phase A gated partner comparisons)
    u64 window_probes = 0;   // U*W
    u64 slow_path_reads = 0; // reads that left the parallel fast mode for the exact sequential chain
    u64 probe_restarts = 0;  // reads redone with verified probes after a 24-bit tag collision
    u64 fast_path_reads = 0;     // reads of phase A certified by the superstring scan (search_fast.cu)
    u64 phase_c_on_device = 0;   // lists / marks / filtering of phase C: 1 device, 2 device with the host's traversal order, 0 host walk
};

struct Timers {   // milliseconds, CUDA events on the context stream
    float ingest = 0, sort_reads = 0, dedupe = 0, build_table = 0, phase_a = 0, phase_b = 0,
          phase_c_dev = 0, phase_c_host = 0, sort_edges = 0, total_device = 0, phase_a_kernel = 0;
};

// peer-memory exchange of the routed probes (shard.cu): this rank's mailbox + the mapped mailboxes of the others
struct Mailbox {
    char *base = nullptr;
    size_t bytes = 0;
    int world = 0, rank = -1;
    u64 cap = 0, ecap = 0;              // windows / entries per (source, owner) segment
    u64 epoch = 0;                      // barriers passed so far (mailbox_barrier)
    char *peer[kMaxWorld] = {};
    bool ipc[kMaxWorld] = {};
};

struct Context {
    Context()
    {
        // everything a context keeps between stages is persistent; stage-local temporaries use `arena`
        d_bases.persistent = d_offsets.persistent = up_d_bases.persistent = up_d_offsets.persistent = up_d_freq.persistent = true;
        raw.persistent = F.persistent = RC.persistent = len.persistent = freq.persistent = true;
        F_loc.persistent = len_loc.persistent = freq_loc.persistent = raw_slice.persistent = entries_loc.persistent = true;
        slots.persistent = entries.persistent = true;
        extR.persistent = extL.persistent = flag5.persistent = cont_max.persistent = explored.persistent = edges.persistent = true;
        rt_queries.persistent = rt_qmap.persistent = rt_wslot.persistent = rt_wentries.persistent = rt_ids.persistent = true;
        rt_redo.persistent = an_resp.persistent = an_entries.persistent = true;
    }
    Arena arena;
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string last_error;
    int min_overlap = 0, h = 0, SW = 0, SWS = 0;     // SW = words per record, SWS = storage stride of F / RC
    // run-time options (sage2gpu_set_option); -1 = take the default / the environment variable
    int opt_low_memory = 0;     // 1: buffers are released as soon as a stage no longer needs them (config #5: 620 M reads on 180 GB)
    int opt_fast_scan = -1;     // phase A: 1 superstring scan first, 0 general kernel only (SAGE2GPU_PA_FAST)
    int opt_read_order = -1;    // phase A schedule: 0 id order, 1 min-hash order (SAGE2GPU_READ_ORDER)
    Counters cnt;
    Timers tm;

    // raw input staged on device
    DevBuf<uint8_t> d_bases;
    DevBuf<int64_t> d_offsets;
    u64 n_input = 0;
    int max_len = 0;
    // streamed upload (sage2gpu_load_begin / _append / _finish): growing device copies of the chunks
    DevBuf<uint8_t> up_d_bases;
    DevBuf<int64_t> up_d_offsets;   // [up_reads + 1], absolute
    u64 up_reads = 0, up_bases = 0;
    bool up_open = false;
    // a saved .reads file (sage2gpu_saved_reads_*): the frequency column of the parsed lines, beside up_d_bases / up_d_offsets
    DevBuf<uint16_t> up_d_freq;
    u64 sr_good = 0, sr_bp = 0;     // sums of FREQ and FREQ * LEN over the lines this context parsed
    cudaEvent_t up_event = nullptr;

    DevBuf<u64> raw;            // [n_input*SW] packed canonical records in input order (step 1, before the sort)
    // unique reads, ids 1..U map to index 0..U-1
    DevBuf<u64> F, RC;          // [U*SWS] records (SW words used, stride SWS = storage_words(SW))
    DevBuf<uint16_t> len, freq; // [U]

    // reads organised by key range over several GPUs (stage_organize_reads with world > 1)
    int rp_rank = 0, rp_world = 1;
    u64 rp_local = 0, rp_first = 0, rp_total = 0;
    u64 rg_total = 0;           // reads of all slices after stage_raw_gather_layout
    // this rank's unique run before it moves into the global arrays (grow-only, kept between calls)
    DevBuf<u64> F_loc;
    DevBuf<uint16_t> len_loc, freq_loc;
    DevBuf<u64> raw_slice;      // this rank's packed slice of a partitioned ingest (the joint array is `raw`)
    DevBuf<u32> entries_loc;    // this rank's shard's entry runs before they move into the joint entries[] array
    bool tb_joint = false;      // the shard was built in its place inside a slot array with room for all shards

    // prefix/suffix table
    DevBuf<u64> slots;          // [cap]
    DevBuf<u32> entries;        // [4U]
    u64 cap = 0;
    int tb_rank = 0, tb_world = 1;   // which key-hash shard the table holds (0 / 1: all keys)
    int tb_shards = 1;               // > 1: the complete table assembled from that many shards (stage_table_gather_*)
    u64 tb_entries = 0;              // entries[] elements in use

    // phase A output
    DevBuf<u64> extR, extL;     // [U] ext_pack
    DevBuf<uint8_t> flag5;      // [U] connections > 300
    DevBuf<u32> cont_max;       // [U] largest (1-based) id whose scan found this read contained
    // phase B output
    DevBuf<uint8_t> explored;   // [U] 0 / 4 / 5 / 6
    // edges
    DevBuf<u64> edges;          // [2*n_edges] (w0,w1) pairs, canonical sorted after finalize
    std::vector<u64> h_edges;   // host copy of final edges (w0,w1 interleaved)
    PinnedBuf pc_stage;         // phase C: the lists of the host traversal land here
    bool have_reads = false, have_table = false, have_phase_a = false, have_phase_b = false, have_graph = false;
    u64 pa_chunk = 0;           // reads per rank in the last phase-A call (partition_chunk)
    int pa_world = 1;
    u64 pa_lo = 0, pa_hi = 0;   // this rank's slice of the reads (sharded phase A)

    // routed probes (shard.cu).  Source side: the current batch
    DevBuf<u64> rt_queries;     // [Q] key hashes or [2Q] keys, one contiguous stream per owner
    DevBuf<u32> rt_qmap;        // [Q] send position -> s * rt_wstride + window
    DevBuf<u64> rt_wslot;       // [rt_n * rt_wstride] answer word of every window of the batch
    DevBuf<u32> rt_wentries;    // entry streams of all owners back to back
    DevBuf<u32> rt_ids;         // list batches: 0-based read indices, ascending
    DevBuf<uint8_t> rt_redo;    // [pa_chunk] reads of the slice that met a tag collision
    u64 rt_n = 0, rt_first = 0, rt_Q = 0, rt_counts[kMaxWorld] = {};
    u32 rt_wstride = 0;
    int rt_what = 0, rt_world = 1, rt_state = 0;     // state: 0 idle, 1 queries out, 2 answers in
    bool rt_is_list = false, rt_exact = false, rt_for_c = false, rt_mailbox = false;
    const u32 *rt_entries_view = nullptr;   // the batch's entry streams: rt_wentries, or the mailbox region read in place
    Mailbox mb;
    // owner side: the answers of the last sage2gpu_shard_answer
    DevBuf<u64> an_resp;
    DevBuf<u32> an_entries;
};

// A file that breaks the grammar of a saved .reads file: `line` = the 1-based line (of the file, or of a context's slice)
struct FormatError : public std::runtime_error {
    u64 line;
    std::string rule;
    FormatError(u64 l, const std::string &r, bool in_slice = false)
        : std::runtime_error("line " + std::to_string(l) + (in_slice ? " of this context's slice: " : ": ") + r), line(l), rule(r) {}
};

// A file that cannot be opened or read
struct IoError : public std::runtime_error {
    explicit IoError(const std::string &m) : std::runtime_error(m) {}
};

// stages (each throws sg::CudaError)
void stage_ingest_ascii(Context &c, const uint8_t *bases, const int64_t *offsets, int64_t n_reads, bool device_resident, int forced_max_len = 0);
void stage_raw_gather_layout(Context &c, int rank, int world, const u64 *counts, void **raw, u64 *first, u64 *total);
void stage_raw_gather_finish(Context &c, u64 total_reads, u64 good_reads, u64 total_bp);
// synth.cu: synthetic paired-end reads generated on the device (measurement aid)
void stage_synth_reads(Context &c, uint8_t *d_bases, int64_t *d_offsets, u64 first_pair, u64 n_pairs, u64 genome_bp, int read_len, float mu, float sigma, u64 seed);
void stage_upload_chunk(Context &c, const uint8_t *bases, const int64_t *offsets, int64_t n_reads);
int stage_uploaded_max_len(Context &c);     // longest read of the streamed upload so far
// parse.cu: record splitting of raw FASTA/FASTQ text on the device; false = irregular layout, nothing appended
bool stage_parse_text_chunk(Context &c, const uint8_t *text, u64 n_bytes, bool final, int &marker, u64 max_records, u64 &consumed, u64 &n_records);
void stage_remove_uploaded(Context &c, u64 first, u64 count);
// parse.cu: a saved .reads file (ReadLoader::loadReadsFromFile, readLoader.cpp:289).  Header: the declared number of reads and the
// byte offset of the body.  Slice: the lines whose first byte lies in [begin, end) of the body, parsed and checked on the device into
// the upload buffers + the frequency column; throws FormatError with the line counted from the slice's first line.
void saved_reads_header(const char *path, u64 &n_reads, u64 &body_offset, u64 &body_bytes);
void stage_parse_saved_reads(Context &c, const char *path, u64 begin, u64 end, u64 &n_lines, int &max_len);
// reads.cu: the parsed lines packed at the stride of max_len (the longest read of all slices) and written as this context's unique run
// (world > 1: F_loc / len_loc / freq_loc, as stage_organize_reads leaves them), then the checks over the complete reads
void stage_pack_saved_reads(Context &c, int rank, int world, int max_len);
void stage_check_saved_reads(Context &c, u64 n_reads, u64 good_reads, u64 total_bp);
void stage_organize_reads(Context &c, int rank = 0, int world = 1);   // world > 1: this rank's key range of the reads only
void stage_reads_gather_layout(Context &c, const u64 *counts, void **F, void **len, void **freq, u64 *first, u64 *total);
void stage_reads_gather_finish(Context &c);
void stage_build_table(Context &c, int rank = 0, int world = 1, bool joint = false);   // key-hash shard `rank` of `world` (SURVEY 8(e)); joint: inside an array with room for all shards
u64 table_shard_slots(u64 unique_reads, int world);     // slots of one key-hash shard of `world` (of the whole table when world = 1)
void stage_table_gather_layout(Context &c, const u64 *entry_counts, void **slots, void **entries, u64 *slots_per_shard, u64 *entries_first);
void stage_table_gather_finish(Context &c, const u64 *entry_counts, const u64 *distinct, const u64 *over);
void stage_phase_a(Context &c, int rank = 0, int world = 1);
void stage_phase_a_import(Context &c, Context &src, int src_rank);   // single-process multi-GPU host: rank src_rank's slice of the phase-A arrays   // rank's slice of the reads; arrays padded to world * chunk
// sharded table (shard.cu, search.cu)
void stage_phase_a_sharded_begin(Context &c, int rank, int world);
void stage_route_begin(Context &c, int what, u64 first, u64 count, int exact, int world, void **queries, u64 *counts);
void stage_shard_answer(Context &c, const void *queries, const u64 *counts_per_source, int exact, int world, void **responses, void **entries,
                        u64 *entry_counts);
void stage_route_finish(Context &c, const void *responses, const void *entries, const u64 *entry_counts);
u64 stage_phase_a_routed(Context &c);
// ... and the same exchange over peer memory (NVLink P2P stores / copies into the ranks' mailboxes)
void stage_mailbox_create(Context &c, int rank, int world, u64 cap_windows, void *ipc_handle_out, void **local_ptr);
void stage_mailbox_open(Context &c, int peer_rank, const void *ipc_handle, void *ptr);
void stage_mailbox_destroy(Context &c);
void stage_mailbox_barrier(Context &c);
void stage_route_post(Context &c, int what, u64 first, u64 count, int exact, u64 *n_reads);
void stage_answer_post(Context &c, int exact, u64 *bytes_sent);
void stage_route_collect(Context &c);
void stage_phase_a_sharded_end(Context &c);
// mapids.cu: step-6 mapping of reads to ids (getIdOfRead, readLoader.cpp:319-353); returns the kernel milliseconds
float stage_map_reads(Context &c, const uint8_t *bases, const int64_t *offsets, int64_t n_reads, bool device_resident, int64_t *ids, uint8_t *good);
void stage_phase_b(Context &c);
void stage_phase_c_and_finalize(Context &c);
// digest.cu: order-sensitive digests of the unique reads / the edge list (parity gate of the measurements)
void stage_digest(Context &c, u64 *reads_digest, u64 *edges_digest);
// device-side text formatters of the reference's -s files (format.cu); false = short write
bool write_reads_text(Context &c, FILE *f);
bool write_graph3_text(Context &c, FILE *f);

}  // namespace sg
