/* sage2gpu.h -- C ABI of libsage2gpu: SAGE2 steps 1-3 (organise reads, prefix/suffix hash table,
 * economy overlap graph) on one NVIDIA B200 (sm_100a).
 *
 * The reference has no plugin / FFI layer: its boundary is the C++ object protocol main.cpp drives
 * (main.cpp:37-132).  Each entry point below names the reference call(s) it replaces; paths are
 * relative to the SAGE2 source tree.  INTEGRATION.md shows the shim a maintainer adds to main.cpp
 * and the makefile link line.
 *
 * Conventions: plain C types, caller-owned host buffers, library-owned device memory, no exceptions
 * across the ABI.  Every function returns 0 on success and a non-zero code on failure;
 * sage2gpu_last_error() then describes the failure (the reference's convention is printError ->
 * log + exit, utils.cpp:36-40; the host shim forwards the string to it).  There is no CPU fallback:
 * without a CUDA device sage2gpu_create() fails.
 *
 * Read ids are the reference's: 1-based ranks of the unique canonical reads in
 * Read::operator< order (readLoader.cpp:11-18,215-260).
 */
#ifndef SAGE2GPU_H
#define SAGE2GPU_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct sage2gpu_ctx sage2gpu_ctx;

enum { SAGE2GPU_OK = 0, SAGE2GPU_ERR_CUDA = 1, SAGE2GPU_ERR_ARG = 2, SAGE2GPU_ERR_STATE = 3, SAGE2GPU_ERR_IO = 4,
       SAGE2GPU_ERR_FORMAT = 5 /* sage2gpu_load_append_text / _bgzf: not the regular 4-line FASTQ / 2-line FASTA layout;
                                  sage2gpu_*bgzf: a BGZF member fails a check;
                                  sage2gpu_*gzip: gzip data fails a check of zlib's inflate / gzread;
                                  sage2gpu_*saved_reads*: the file breaks the grammar of a saved .reads file */ };

/* Log counters of the reference (readLoader.cpp:164-169,257; hashTable.cpp:86,124;
 * economyGraph.cpp:485-487,569-571) plus the workload sizes the roofline needs. */
typedef struct {
    uint64_t total_reads, good_reads, unique_reads, total_bp, avg_len;
    uint64_t hash_len, distinct_keys, keys_over_threshold, table_capacity;
    uint64_t contained_ext, contained_size, left_to_explore;
    uint64_t edges_phase_b, candidates_c, edges_inserted_c, transitive_removed;
    uint64_t n_edges;
    uint64_t compare_calls;     /* V of SURVEY 8(d): gated partner comparisons in phase A */
    uint64_t window_probes;     /* U*W table probes in phase A */
    uint64_t slow_path_reads;   /* reads whose extension chain ran hit by hit (ambiguity / multi-hit windows) */
    uint64_t record_words;      /* 64-bit words per packed read record */
    uint64_t probe_restarts;    /* reads redone with verified probes after a tag collision */
    uint64_t phase_c_on_device; /* phase C lists / marks / filtering: 1 on the device (order-independent input), 2 on the device with
                                   the traversal order from the host, 0 whole walk on the host */
    uint64_t fast_path_reads;   /* phase-A reads certified by the superstring scan (the rest took the hit-by-hit kernel) */
} sage2gpu_counters;

/* Stage times in milliseconds (CUDA events on the context's stream; host part by steady_clock). */
typedef struct {
    float ingest, sort_reads, build_table, phase_a, phase_b, phase_c_dev, phase_c_host, sort_edges, total;
    float phase_a_kernel;   /* the phase-A search kernel alone (events around the launch) */
} sage2gpu_timers;

/* One undirected edge as OverlapGraph::convertGraph creates it (overlapGraph.cpp:84-159):
 * from < to; `type` and `delta` describe from->to, `delta_twin` the twin to->from
 * (type of the twin = reverseEdgeType(type), utils.cpp:212-219). */
typedef struct {
    uint64_t from, to;
    uint32_t type, delta, delta_twin, reserved;
} sage2gpu_edge;

/* replaces: object construction in main.cpp:44,76,108.  device = CUDA ordinal. */
int  sage2gpu_create(sage2gpu_ctx **ctx, int device);
void sage2gpu_destroy(sage2gpu_ctx *ctx);
const char *sage2gpu_last_error(const sage2gpu_ctx *ctx);

/* replaces: ReadLoader::readDatasetInBytes' per-read work + organizeReads
 * (readLoader.cpp:133-260; isGoodRead utils.cpp:144, insertReadIntoList readLoader.cpp:179).
 * `bases` = the read sequences concatenated (ASCII, any case), read r = bases[offsets[r],
 * offsets[r+1]).  Host buffers (pinned memory makes the upload asynchronous).  Reads with
 * length <= min_overlap or a non-ACGT character are dropped exactly like the reference does.  Limit of this build: reads
 * of up to 1016 bases (the reference has none); a longer read makes the call fail rather than renumber the reads. */
int sage2gpu_load_reads(sage2gpu_ctx *ctx, const uint8_t *bases, const int64_t *offsets,
                        int64_t n_reads, int min_overlap);
/* Same, with both buffers already resident in this context's device memory. */
int sage2gpu_load_reads_device(sage2gpu_ctx *ctx, const uint8_t *d_bases, const int64_t *d_offsets,
                               int64_t n_reads, int min_overlap);

/* The same as sage2gpu_load_reads, streamed: the reference reads its input record by record
 * (readLoader.cpp:146-160); the host parser fills one pinned chunk while the previous one is uploaded.
 * offsets has n_reads+1 entries relative to `bases` (read r = bases[offsets[r], offsets[r+1])).  A chunk's
 * buffers may be reused as soon as a LATER call to _append or _finish has returned.  _finish runs the
 * filter / pack / sort / dedupe of organizeReads. */
int sage2gpu_load_begin(sage2gpu_ctx *ctx, int min_overlap);
int sage2gpu_load_append(sage2gpu_ctx *ctx, const uint8_t *bases, const int64_t *offsets, int64_t n_reads);
int sage2gpu_load_finish(sage2gpu_ctx *ctx);
/* The same with the record splitting on the device (replaces the per-record work of FastAQReader::getNextRead,
 * fastAQReader.cpp:16-45, for regular files): `text` is a piece of a FASTA / FASTQ file (already inflated if it was
 * gzip) that starts at a record boundary.  Every complete record in it (at most max_records) is appended;
 * *consumed tells how many bytes they took -- the caller prepends the rest to the next piece; is_final marks
 * the last piece.  *marker is 0 before the first piece of a file and carries '@' / '>' afterwards.  Returns
 * SAGE2GPU_ERR_FORMAT, with nothing appended, when the piece is not in the regular 4-line FASTQ / 2-line
 * FASTA layout (multi-line records, blank lines, empty sequences, a truncated tail ...): the caller then
 * parses that text sequentially and uses sage2gpu_load_append.  The buffer may be reused on return. */
int sage2gpu_load_append_text(sage2gpu_ctx *ctx, const uint8_t *text, uint64_t n_bytes, int is_final, int *marker,
                              uint64_t max_records, uint64_t *consumed, uint64_t *n_records);
/* The same for a piece of a BGZF-compressed file (htslib's bgzip: gzip members of at most 64 KiB of text, each with a `BC`
 * extra subfield holding BSIZE), inflated on the device (replaces FastAQReader::getNextRead, fastAQReader.cpp:16-45, over
 * kseq + gzread).  bgzf[0, n_bytes) holds whole members; their text follows prefix[0, prefix_bytes) (host text: what the
 * previous piece did not consume, which may have gone to another context), and that text is split exactly as
 * sage2gpu_load_append_text splits it, with the same is_final, *marker, max_records, *n_records and *consumed (bytes of that
 * text, prefix included).  *rest_bytes = the text not consumed; its first min(*rest_bytes, rest_capacity) bytes are copied to
 * `rest` -- the prefix of the next piece.  Every member's CRC32 and ISIZE are checked.  Returns SAGE2GPU_ERR_FORMAT with
 * nothing appended when a member fails a check (*bad_member = its index in the piece, sage2gpu_last_error names it and the
 * rule; the context stays usable) or when the text is irregular (*bad_member = -1: parse it sequentially, as with
 * _append_text).  The buffers may be reused on return. */
int sage2gpu_load_append_bgzf(sage2gpu_ctx *ctx, const uint8_t *prefix, uint64_t prefix_bytes, const uint8_t *bgzf, uint64_t n_bytes,
                              int is_final, int *marker, uint64_t max_records, uint64_t *consumed, uint64_t *n_records, uint8_t *rest,
                              uint64_t rest_capacity, uint64_t *rest_bytes, int64_t *bad_member);
/* The BGZF members of bgzf[0, n_bytes) inflated on the device into text[0, *text_bytes) (host buffers; *text_bytes = the sum of
 * their ISIZEs, set even when text_capacity is too small, which fails with SAGE2GPU_ERR_STATE).  Checks and *bad_member as
 * above.  *kernel_ms (may be NULL) = the inflate kernel alone. */
int sage2gpu_inflate_bgzf(sage2gpu_ctx *ctx, const uint8_t *bgzf, uint64_t n_bytes, uint8_t *text, uint64_t text_capacity, uint64_t *text_bytes,
                          int64_t *bad_member, float *kernel_ms);
/* Where a piece of an ordinary gzip stream (single-member, or members concatenated, as gzip / pigz write them) continues.  All
 * zeros before the first piece.  A piece hands this to the next one, whichever context decodes it. */
typedef struct {
    uint64_t offset;          /* compressed byte offset (in the file) of the byte the next piece starts with */
    uint64_t member_offset;   /* compressed offset of the current member's header */
    uint64_t member_bytes;    /* text of the current member so far (its ISIZE is this mod 2^32) */
    uint32_t bit;             /* the next DEFLATE block starts at this bit (0-7) of that byte */
    uint32_t in_member;       /* 1: the next piece starts at a block of the current member; 0: at a member header or the end */
    uint32_t crc;             /* CRC32 of the current member's text so far */
    uint32_t window_bytes;    /* bytes of the current member's text at the end of window[] (at most 32768) */
    uint32_t done;            /* the stream has ended: a trailer followed by the end of the file or by bytes that are not a gzip
                                 header (zlib ignores them) */
    uint32_t reserved;
    uint8_t window[32768];    /* the current member's last text, ending at window[32767] */
} sage2gpu_gzip_state;
/* The same as sage2gpu_load_append_bgzf for a piece of an ordinary gzip file, inflated on the device (replaces
 * FastAQReader::getNextRead, fastAQReader.cpp:16-45, over kseq + gzread, whose text this equals byte for byte).  gz[0, n_bytes)
 * are the compressed bytes from state->offset on; is_final says that they reach the end of the file.  The piece is cut at
 * DEFLATE block starts found on the device, its ranges inflated at once and stitched; at most max(text_bound, one range of
 * blocks) bytes of text are inflated, after the host prefix, and split as _load_append_text splits them (prefix, is_final of
 * the splitter = the stream ended in this piece, *marker, max_records, *consumed, *n_records, rest as for _bgzf).  *state moves
 * to where the next piece starts and *in_consumed = the compressed bytes it moved past: 0 when the piece holds no complete
 * block (pass more bytes).  Every member's CRC32 and ISIZE are checked.  Returns SAGE2GPU_ERR_FORMAT with nothing appended and
 * *state unchanged when the data fails a check (*bad_offset = the compressed offset of the member -- header, CRC, ISIZE,
 * truncated trailer -- or of the block that broke a DEFLATE rule; sage2gpu_last_error names it and the rule; the context
 * stays usable) or when the text is irregular (*bad_offset = -1: parse it sequentially).  The buffers may be reused on return. */
int sage2gpu_load_append_gzip(sage2gpu_ctx *ctx, const uint8_t *prefix, uint64_t prefix_bytes, const uint8_t *gz, uint64_t n_bytes,
                              int is_final, uint64_t text_bound, sage2gpu_gzip_state *state, int *marker, uint64_t max_records,
                              uint64_t *consumed, uint64_t *n_records, uint8_t *rest, uint64_t rest_capacity, uint64_t *rest_bytes,
                              uint64_t *in_consumed, int64_t *bad_offset);
/* A whole gzip stream gz[0, n_bytes) inflated on the device into text[0, *text_bytes) (host buffers; fails with
 * SAGE2GPU_ERR_STATE when the text is larger than text_capacity, *text_bytes then being the text inflated so far).  Checks and
 * *bad_offset as above.  *kernel_ms = the device kernels alone, *ranges = ranges decoded (all passes, false candidates
 * included), *confirmed = ranges whose text was kept (the confirmed chains of all pieces), *rejected = block-start candidates
 * found false; each may be NULL. */
int sage2gpu_inflate_gzip(sage2gpu_ctx *ctx, const uint8_t *gz, uint64_t n_bytes, uint8_t *text, uint64_t text_capacity, uint64_t *text_bytes,
                          int64_t *bad_offset, float *kernel_ms, uint64_t *ranges, uint64_t *confirmed, uint64_t *rejected);
/* Reads appended since sage2gpu_load_begin; removal of the appended reads [first, first + count) (the reference
 * stops a two-file data set when the shorter mate file ends, inputReader.cpp:26-49). */
int sage2gpu_load_count(sage2gpu_ctx *ctx, uint64_t *n_reads);
int sage2gpu_load_remove(sage2gpu_ctx *ctx, uint64_t first, uint64_t count);
/* Page-locked host memory for the buffers above (plain malloc'ed memory works too, synchronously). */
void *sage2gpu_host_alloc(uint64_t n_bytes);
void sage2gpu_host_free(void *p);

/* ---- Restart from a saved .reads file ----------------------------------------------------------------------------------
 * replaces: ReadLoader::loadReadsFromFile (readLoader.cpp:289), which SAGE2 -m 2 / -m 3 calls.  The file is what
 * ReadLoader::saveReadsInFile writes (readLoader.cpp:270-287, and sage2gpu_write_reads byte for byte): a line with the number of
 * reads U, then U lines "FREQ	LEN	F	R
".  Accepted is exactly that: FREQ a decimal in 0..65535, LEN in 1..1016 (the limit of
 * this build) and greater than min_overlap, both without leading zeros; F and R of LEN upper-case ACGT characters, R the reverse
 * complement of F, F <= R (the strand insertReadIntoList keeps, readLoader.cpp:195); the F records strictly increasing in
 * Read::operator< order (line n + 1 is read id n); U lines.  Anything else -- a truncated file, lower case, N, '
', extra lines,
 * gzip -- fails with SAGE2GPU_ERR_FORMAT and nothing loaded; sage2gpu_last_error names the 1-based line and the rule.  Parsing and
 * checks run on the device, in pieces of the file.  After success the context is as after sage2gpu_load_finish: unique_reads = U,
 * good_reads = total_reads = sum of FREQ, total_bp = sum of FREQ * LEN, avg_len = total_bp / good_reads (0 when the sum is 0).
 * Those equal a run from the input files unless a read occurred 65,536 times or more: its FREQ is the uint16_t count wrapped
 * (readLoader.cpp:234), so the sums count it modulo 65,536. */
int sage2gpu_load_saved_reads(sage2gpu_ctx *ctx, const char *path, int min_overlap);
/* The same over several contexts (body = the file without its first line):
 *   saved_reads_info        U (*n_reads) and the size of the body in bytes
 *   saved_reads_slice       the lines whose first byte lies in [byte_begin, byte_end) of the body, parsed and checked on this
 *                           context; *n_lines, *max_read_length = its longest read.  On SAGE2GPU_ERR_FORMAT *bad_line = the line
 *                           counted from the slice's first line (its file line = 1 + the lines of the slices before + *bad_line)
 *   [maximum over the contexts]
 *   saved_reads_pack        the slice packed at the record stride of max_read_length (the longest read of ALL slices) as this
 *                           context's unique run, as sage2gpu_organize_partition leaves it (world = 1: the reads themselves);
 *                           *unique_local = its lines, *good_reads / *total_bp = its sums of FREQ and FREQ * LEN
 *   [world > 1: sage2gpu_reads_gather_layout, the all-gather, sage2gpu_reads_gather_finish]
 *   saved_reads_finish      the sums over the contexts: checks the count against U and the order of the complete reads (pairs
 *                           that straddle two slices too) and sets the counters; on SAGE2GPU_ERR_FORMAT *bad_line = the file line.
 * sage2gpu_load_saved_reads = info + slice(0, body) + pack(0, 1) + finish. */
int sage2gpu_saved_reads_info(sage2gpu_ctx *ctx, const char *path, uint64_t *n_reads, uint64_t *body_bytes);
int sage2gpu_saved_reads_slice(sage2gpu_ctx *ctx, const char *path, int min_overlap, uint64_t byte_begin, uint64_t byte_end, uint64_t *n_lines,
                               int *max_read_length, uint64_t *bad_line);
int sage2gpu_saved_reads_pack(sage2gpu_ctx *ctx, int rank, int world, int max_read_length, uint64_t *unique_local, uint64_t *good_reads,
                              uint64_t *total_bp);
int sage2gpu_saved_reads_finish(sage2gpu_ctx *ctx, uint64_t n_reads, uint64_t good_reads, uint64_t total_bp, uint64_t *bad_line);

/* replaces: HashTable::hashPrefixesAndSuffix (hashTable.cpp:70-128) */
int sage2gpu_build_hash_table(sage2gpu_ctx *ctx);

/* replaces: EconomyGraph::buildInitialOverlapGraph + buildOverlapGraphEconomy + sortEconomyGraph
 * (economyGraph.cpp:37-574,896-913) and the edge selection of OverlapGraph::convertGraph
 * (overlapGraph.cpp:93-112).  Leaves the canonical edge list on the device; sage2gpu_get_edges[_packed],
 * sage2gpu_write_graph3 bring it to the host. */
int sage2gpu_build_overlap_graph(sage2gpu_ctx *ctx);

/* Read-only view of the table this context holds (after any build_hash_table* call, and after table_gather_finish):
 * device pointers to the slot index (*n_slots uint64 words, `shards` key-hash shards of *sectors_per_shard sectors of 4 slots
 * each, back to back) and to the entry runs (*n_entries uint32), as core.cuh lays them out.  A context of the sharded layout
 * (build_hash_table_shard) holds one shard: the keys it owns. */
int sage2gpu_table_view(sage2gpu_ctx *ctx, const void **slots, uint64_t *n_slots, const void **entries, uint64_t *n_entries,
                        uint64_t *sectors_per_shard, uint64_t *shards);

/* Multi-GPU form of the same step (SURVEY.md 8(e)): phase A is independent per read
 * (the reference's `omp for`, economyGraph.cpp:71), so with the reads and the table present on every GPU rank
 * `rank` of `world` searches only read ids [rank*chunk, (rank+1)*chunk), chunk = ceil(U/world).
 * sage2gpu_phase_a_buffers exposes the device arrays (length world*chunk; uint64 extension records of
 * rightExtension / leftExtension, uint8 "connections > 300" flags, uint32 largest id that contains the
 * read) for the one exchange step -- all-gather of the first three, all-reduce(MAX) of the last, e.g.
 * NCCL through sage2_b200/multi.py -- after which sage2gpu_finish_graph runs phases B and C and the
 * canonical edge sort.  build_overlap_graph == phase_a_partition(0, 1) + finish_graph. */
int sage2gpu_phase_a_partition(sage2gpu_ctx *ctx, int rank, int world);
int sage2gpu_phase_a_buffers(sage2gpu_ctx *ctx, void **right_ext, void **left_ext, void **over_limit, void **contained_by,
                             uint64_t *reads_per_rank, uint64_t *unique_reads);
int sage2gpu_finish_graph(sage2gpu_ctx *ctx);

/* ---- Several GPUs, every stage partitioned (SURVEY.md 8(e)) ----------------------------------------------------------
 * The packed reads end up replicated on every GPU, as north_star asks, but no GPU does another GPU's work:
 *
 *   load_reads_partition(rank, world)   organizeReads (readLoader.cpp:215-260) for the reads whose leading bases fall into
 *                                       this rank's key range: every rank sees the whole input, derives the same splitters
 *                                       from a histogram of the leading 6 bases and sorts + dedupes only its range;
 *                                       *unique_local = its number of unique reads.  Equal reads share a range, so the
 *                                       ranks' runs concatenate to the global sorted order (read ids stay the reference's).
 *   [all-gather of the counts]          reads_gather_layout(counts): device arrays of the total size with this rank's run
 *                                       in its place (records: uint64 x record_stride_words per read; lengths,
 *                                       frequencies: uint16); [first, first + counts[rank]) is this rank's id range
 *   [all-gather of the three arrays, variable block sizes]   reads_gather_finish(): reverse complements, done.
 *   build_hash_table_part(rank, world)  hashPrefixesAndSuffix (hashTable.cpp:70-128) for the keys this rank owns, built in its
 *                                       place inside a slot array with room for all shards;
 *   table_shard_info, [all-gather of the entry counts], table_gather_layout(entry_counts): room for all shards back to
 *                                       back (slots: slots_per_shard uint64 per shard; entries: uint32), own shard in place
 *   [all-gather of both arrays]         table_gather_finish(): the complete table on every GPU; probes stay local
 *   phase_a_partition(rank, world) + exchange of phase_a_buffers + finish_graph as before.
 * The exchanges are the host's (NCCL through sage2_b200/multi.py, or peer copies inside one process). */
int sage2gpu_load_reads_partition(sage2gpu_ctx *ctx, const uint8_t *bases, const int64_t *offsets, int64_t n_reads, int min_overlap,
                                  int on_device, int rank, int world, uint64_t *unique_local);
/* The same with the INGEST partitioned too (inputs that no single GPU should hold as characters, e.g. config #5):
 *   pack_slice(slice, max_read_length)  isGoodRead + canonical orientation + 2-bit pack (readLoader.cpp:146-213) of this
 *                                       rank's slice of the input; max_read_length = longest read of the WHOLE read set
 *                                       (it fixes the record stride on every rank); sums of *good_reads / *total_bp over
 *                                       the ranks are the read set's counters
 *   [all-gather of the slice sizes]     raw_gather_layout(counts): room for the packed records of all slices, own slice in place
 *   [all-gather of the records, record_words uint64 per read; all-reduce of the counters]   raw_gather_finish(totals)
 *   organize_partition(rank, world)     as load_reads_partition from here on. */
int sage2gpu_pack_slice(sage2gpu_ctx *ctx, const uint8_t *bases, const int64_t *offsets, int64_t n_reads, int min_overlap, int on_device,
                        int max_read_length, uint64_t *good_reads, uint64_t *total_bp, uint64_t *record_words);
int sage2gpu_raw_gather_layout(sage2gpu_ctx *ctx, int rank, int world, const uint64_t *counts, void **records, uint64_t *first, uint64_t *total);
int sage2gpu_raw_gather_finish(sage2gpu_ctx *ctx, uint64_t total_reads, uint64_t good_reads, uint64_t total_bp);
int sage2gpu_organize_partition(sage2gpu_ctx *ctx, int rank, int world, uint64_t *unique_local);
/* Measurement aid (no reference counterpart): pairs [first_pair, first_pair + n_pairs) of a synthetic error-free paired-end
 * read set (uniform-random genome of genome_bp bases that is a pure function of the seed, mates interleaved, insert size
 * ~ N(insert_mean, insert_sd) clipped to >= 2 * read_length) written as characters into DEVICE buffers: d_bases
 * (2 * n_pairs * read_length bytes), d_offsets (2 * n_pairs + 1).  Any rank can generate any slice. */
int sage2gpu_synth_reads(sage2gpu_ctx *ctx, uint8_t *d_bases, int64_t *d_offsets, uint64_t first_pair, uint64_t n_pairs, uint64_t genome_bp,
                         int read_length, float insert_mean, float insert_sd, uint64_t seed);
int sage2gpu_reads_gather_layout(sage2gpu_ctx *ctx, const uint64_t *counts, void **records, void **lengths, void **frequencies,
                                 uint64_t *first, uint64_t *total, uint64_t *record_stride_words);
int sage2gpu_reads_gather_finish(sage2gpu_ctx *ctx);
int sage2gpu_build_hash_table_part(sage2gpu_ctx *ctx, int rank, int world);
int sage2gpu_table_shard_info(sage2gpu_ctx *ctx, uint64_t *slots, uint64_t *entries, uint64_t *distinct_keys, uint64_t *keys_over_threshold);
int sage2gpu_table_gather_layout(sage2gpu_ctx *ctx, const uint64_t *entry_counts, void **slots, void **entries, uint64_t *slots_per_shard,
                                 uint64_t *entries_first);
int sage2gpu_table_gather_finish(sage2gpu_ctx *ctx, const uint64_t *entry_counts, const uint64_t *distinct_keys,
                                 const uint64_t *keys_over_threshold);

/* ---- One process, several GPUs (host/sage2gpu_main.cpp --devices): the exchanges of the partitioned build as peer copies ----
 * load_finish_packed   = sage2gpu_load_finish without organizeReads: the streamed upload is filtered and packed
 *                        (readLoader.cpp:146-213) and stays this context's slice, as after pack_slice; *max_read_length is what
 *                        the other contexts pass to pack_slice (with 0 reads) before raw_gather_layout
 * peer_copy            bytes from src's device memory into dst's (cudaMemcpyPeer): the all-gathers between the *_gather_layout
 *                        and *_gather_finish calls
 * phase_a_import       rank src_rank's slice of the phase-A arrays of `src` into `ctx` (+ element-wise maximum of the
 *                        containment ids): the exchange of sage2gpu_phase_a_buffers */
int sage2gpu_load_finish_packed(sage2gpu_ctx *ctx, uint64_t *n_reads, int *max_read_length, uint64_t *good_reads, uint64_t *total_bp);
/* A streamed upload spread over several contexts (each received a part of the input through _append / _append_text):
 *   load_max_length      the longest read appended to this context since sage2gpu_load_begin (nothing is packed)
 *   [maximum over the contexts]
 *   load_finish_slice    = pack_slice on the uploaded reads: filtered and packed at the record stride of max_read_length (the
 *                        longest read of the WHOLE read set), this context's slice for raw_gather_layout; *n_reads = its reads */
int sage2gpu_load_max_length(sage2gpu_ctx *ctx, int *max_read_length);
int sage2gpu_load_finish_slice(sage2gpu_ctx *ctx, int max_read_length, uint64_t *n_reads, uint64_t *good_reads, uint64_t *total_bp,
                               uint64_t *record_words);
/* After sage2gpu_reads_gather_finish (or any load that organised the reads): the bytes of the table this context would hold
 * with `world` contexts, replicated (build_hash_table_part + table_gather_*: all shards) or sharded (build_hash_table_shard: one
 * shard).  Slot bytes are exact; entry bytes are an upper bound (4 entries per unique read).  *device_free_bytes (may be NULL) =
 * cudaMemGetInfo's free memory of the context's GPU, shared by all contexts on it.  For choosing between the two layouts. */
int sage2gpu_table_bytes(sage2gpu_ctx *ctx, int world, uint64_t *replicated_slot_bytes, uint64_t *replicated_entry_bytes,
                         uint64_t *sharded_slot_bytes, uint64_t *sharded_entry_bytes, uint64_t *device_free_bytes);
int sage2gpu_peer_copy(sage2gpu_ctx *dst, void *dst_ptr, sage2gpu_ctx *src, const void *src_ptr, uint64_t n_bytes);
int sage2gpu_phase_a_import(sage2gpu_ctx *ctx, sage2gpu_ctx *src, int src_rank);

/* ---- The table sharded by key hash (SURVEY.md 8(e), north_star) ---------------------------------------------------
 * The reads stay on every GPU; shard `rank` of `world` indexes only the keys whose hash it owns, so the table of a
 * data set is spread over the GPUs of the box.  A window probe of HashTable::hashTableSearch (hashTable.cpp:193-231)
 * becomes a query routed to the owner of its key (all-to-all between the ranks, e.g. NCCL through
 * sage2_b200/multi.py; this library only fills and consumes the device buffers):
 *
 *   build_hash_table_shard                         replaces hashPrefixesAndSuffix (hashTable.cpp:70-128) for one shard
 *   phase_a_sharded_begin                          this rank's slice [first, first+count) of the unique reads (0-based)
 *   per batch of the slice:
 *     route_begin(what=0, first, count, exact=0)   window keys of the batch bucketed by owner: `queries` = world
 *                                                  contiguous streams (counts[g] queries for owner g; a query is one
 *                                                  uint64 key hash, or two uint64 = the 128-bit key when exact)
 *     [all-to-all]  shard_answer                   the owner's answers: one uint64 per received query, same order,
 *                                                  + one stream of uint32 bucket entries per source (entry_counts[s])
 *     [all-to-all]  route_finish                   answers back at the source, in the order the queries were sent;
 *                                                  entry streams of owner 0, 1, .. back to back
 *     phase_a_routed                               the phase-A kernel of buildInitialOverlapGraph (economyGraph.cpp:64-452)
 *                                                  on the batch; *n_redo = reads that met a 24-bit tag collision
 *   if any rank has such reads: route_begin(what=2, exact=1) .. phase_a_routed once more (verified probes,
 *                                                  hashTable.cpp:203-220), then phase_a_sharded_end
 *   exchange of the phase-A arrays (sage2gpu_phase_a_buffers), sage2gpu_phase_b,
 *   route_begin(what=1, exact=1) .. route_finish for the reads left for phase C (insertAllEdgesOfRead,
 *   economyGraph.cpp:580-638), sage2gpu_finish_graph.
 * counts / entry_counts arrays have `world` elements (world <= 64); all buffers handed out are device memory owned by
 * the context and stay valid until the next call of the same function. */
int sage2gpu_build_hash_table_shard(sage2gpu_ctx *ctx, int rank, int world);
int sage2gpu_phase_a_sharded_begin(sage2gpu_ctx *ctx, int rank, int world, uint64_t *first, uint64_t *count);
int sage2gpu_route_begin(sage2gpu_ctx *ctx, int what, uint64_t first, uint64_t count, int exact, int world, void **queries,
                         uint64_t *counts, uint64_t *n_reads);
int sage2gpu_shard_answer(sage2gpu_ctx *ctx, const void *queries, const uint64_t *counts_per_source, int exact, int world,
                          void **responses, void **entries, uint64_t *entry_counts);
int sage2gpu_route_finish(sage2gpu_ctx *ctx, const void *responses, const void *entries, const uint64_t *entry_counts);
int sage2gpu_phase_a_routed(sage2gpu_ctx *ctx, uint64_t *n_redo);
int sage2gpu_phase_a_sharded_end(sage2gpu_ctx *ctx);
/* The same exchange over PEER MEMORY (NVLink / NVSwitch P2P) instead of an all-to-all of the host: every rank owns a
 * "mailbox" in its device memory which the other ranks map (CUDA IPC between processes: hand the 64-byte
 * ipc_handle_out of mailbox_create to the other ranks and pass it to their mailbox_open; inside one process pass
 * *local_ptr instead: a mailbox on another GPU gets peer access enabled, and mailbox_open fails when the two GPUs cannot
 * access each other's memory).  The mailbox holds, per peer, room for the windows of max_reads_per_batch reads.
 *   route_post     = route_begin, but the routing kernel stores every query straight into its owner's mailbox
 *   [barrier between the ranks]
 *   answer_post    = shard_answer out of the own mailbox; answers and bucket entries are copied into the sources' mailboxes
 *   [barrier between the ranks]
 *   route_collect  = route_finish out of the own mailbox
 * No sizes travel ahead of the data and the host moves nothing.  *bytes_sent = bytes this rank put into other ranks' memory. */
int sage2gpu_mailbox_create(sage2gpu_ctx *ctx, int rank, int world, uint64_t max_reads_per_batch, void *ipc_handle_out, void **local_ptr);
int sage2gpu_mailbox_open(sage2gpu_ctx *ctx, int peer_rank, const void *ipc_handle, void *ptr);
/* The barrier between the three steps, on the device: every rank stores its barrier count into the peers' mailboxes and
 * waits for theirs (all ranks must call it the same number of times).  A peer that never arrives ends the wait with an
 * error after 60 s (environment SAGE2GPU_BARRIER_TIMEOUT_S); the mailbox is released then and has to be created again. */
int sage2gpu_mailbox_barrier(sage2gpu_ctx *ctx);
int sage2gpu_route_post(sage2gpu_ctx *ctx, int what, uint64_t first, uint64_t count, int exact, uint64_t *n_reads, uint64_t *bytes_sent);
int sage2gpu_answer_post(sage2gpu_ctx *ctx, int exact, uint64_t *bytes_sent);
int sage2gpu_route_collect(sage2gpu_ctx *ctx);

/* Phase B alone (economyGraph.cpp:455-480); sage2gpu_finish_graph skips it when it already ran. */
int sage2gpu_phase_b(sage2gpu_ctx *ctx);

/* All three steps back to back (main.cpp:37-132 without the file I/O). */
int sage2gpu_run_steps123(sage2gpu_ctx *ctx, const uint8_t *bases, const int64_t *offsets,
                          int64_t n_reads, int min_overlap);

/* Measurement aid (no reference counterpart): GB/s this GPU sustains on uniformly random, independent
 * `granule_bytes` (16/32/64) gathers over `footprint_bytes` of device memory -- the random-sector
 * roofline of the probe / partner-fetch traffic (SURVEY.md 8(d)).  mode 0: 128-bit loads; 1: 256-bit loads
 * (granule 32/64); 2: a 64-byte granule fetched by a lane pair, one 256-bit load each. */
int sage2gpu_measure_gather(sage2gpu_ctx *ctx, uint64_t footprint_bytes, int granule_bytes, uint64_t n_loads, int mode, double *gbps);

/* Parity gate of the measurements (no reference counterpart): order-sensitive 64-bit digests of the resident unique
 * reads (what ReadLoader::saveReadsInFile would write, readLoader.cpp:270-287: id, frequency, length, forward bases)
 * and of the canonical edge list (what OverlapGraph::saveOverlapGraphInFile would write, overlapGraph.cpp:338-369:
 * position, from, to, type, both overhangs).  tests/digest.py computes the same sums from the reference's own files.
 * Either pointer may be NULL. */
int sage2gpu_digest(sage2gpu_ctx *ctx, uint64_t *reads_digest, uint64_t *edges_digest);

/* Run-time options.  "read_order": schedule of the phase-A search (results do not depend on it): 0 = id order,
 * 1 = minimizer order (reads that share bases are searched together, so slot sectors and partner records hit L2),
 * -1 = the default: minimizer order when the records and the slot index take 1 GiB or more, id order below.  "low_memory": 1 = the large buffers are released (and returned to the driver) as soon as no later stage of the step
 * needs them -- the packed input after organizeReads, the table before the edge sort; 2 = the workspace too, after every
 * call (for read sets near the capacity of the GPU).  Switched on when the reads are already organised (and gathered), it
 * releases at once what it would have released by then: the packed input, the context's packed slice and unique run, the
 * workspace.  "fast_scan": 1 = phase A tries the superstring scan first (default), 0 = hit-by-hit kernel only. */
int sage2gpu_set_option(sage2gpu_ctx *ctx, const char *name, int64_t value);

int sage2gpu_get_counters(const sage2gpu_ctx *ctx, sage2gpu_counters *out);
/* Number of CUDA kernels this library has launched in this process so far (monotonic). */
uint64_t sage2gpu_kernel_launches(void);
int sage2gpu_get_timers(const sage2gpu_ctx *ctx, sage2gpu_timers *out);
/* The cudaStream_t every kernel of this context is launched on (for external CUDA-event timing). */
void *sage2gpu_stream(const sage2gpu_ctx *ctx);

/* replaces: what steps 4-7 read through ReadLoader::getRead (readLoader.cpp:309): for ids 1..U the
 * length, frequency and both packed strands in the REFERENCE byte layout (utils.cpp:96-119).
 * byte_off has U+1 entries (byte_off[i-1] = start of read i); fwd/rc need byte_off[U] bytes
 * (query with sage2gpu_reads_bytes). */
int sage2gpu_reads_bytes(const sage2gpu_ctx *ctx, uint64_t *n_bytes);
int sage2gpu_get_reads(sage2gpu_ctx *ctx, uint16_t *length, uint16_t *frequency, uint64_t *byte_off,
                       uint8_t *fwd, uint8_t *rc);

/* replaces: ReadLoader::getIdOfRead (readLoader.cpp:319-353) for a whole batch of reads, as step 6 uses it behind
 * isGoodRead (MatePair::processMatePairs, matePair.cpp:176-181).  Input like sage2gpu_load_reads (host buffers, or
 * device buffers when on_device != 0).  ids[r] (host) = +id when read r itself is the stored orientation, -id when
 * its reverse complement is (a read equal to its reverse complement gives -id, readLoader.cpp:325-334), 0 when it is
 * not among the unique reads; good[r] (host, may be NULL) = isGoodRead(read r, min_overlap) -- the reference never
 * looks a bad read up, its id is reported as 0.  *kernel_ms (may be NULL) = the lookup kernel alone. */
int sage2gpu_map_reads(sage2gpu_ctx *ctx, const uint8_t *bases, const int64_t *offsets, int64_t n_reads, int on_device,
                       int64_t *ids, uint8_t *good, float *kernel_ms);

/* Phase A / B state for inspection: packed extension records (id | type<<32 | overhang<<33) of
 * rightExtension / leftExtension (economyGraph.cpp:46-47) and exploredReads after phase B. */
int sage2gpu_get_extensions(sage2gpu_ctx *ctx, uint64_t *right_ext, uint64_t *left_ext, uint8_t *explored);

/* replaces: the economyGraphList hand-over to convertGraph.  capacity in edges; *n_edges receives the
 * total (call with out=NULL to size).  Order = the order convertGraph creates / .graph3 lists them. */
int sage2gpu_get_edges(sage2gpu_ctx *ctx, sage2gpu_edge *out, uint64_t capacity, uint64_t *n_edges);

/* Same list, undecoded, copied straight into the caller's (ideally pinned) buffer: two 64-bit words per
 * edge, w0 = from << 32 | to, w1 = type << 20 | delta; the twin's delta is len(from) - (len(to) - delta)
 * (overlapGraph.cpp:147).  capacity in edges. */
int sage2gpu_get_edges_packed(sage2gpu_ctx *ctx, uint64_t *out, uint64_t capacity, uint64_t *n_edges);

/* replaces: ReadLoader::saveReadsInFile (readLoader.cpp:270-287) and
 * OverlapGraph::saveOverlapGraphInFile (overlapGraph.cpp:338-369): the reference's -s text formats,
 * byte for byte, so that `SAGE2 -m 4 -i <prefix>` continues from them. */
int sage2gpu_write_reads(sage2gpu_ctx *ctx, const char *path);
int sage2gpu_write_graph3(sage2gpu_ctx *ctx, const char *path);
/* No reference counterpart: the same reads and edges as one GFA 1.0 file, formatted on the device (for Bandage, gfatools,
 * vg and other readers of the standard format).  Exactly these bytes, with U = unique reads and ids 1..U as in .reads:
 *   H<TAB>VN:Z:1.0<LF>
 *   S<TAB><id><TAB><F><TAB>LN:i:<len><TAB>RC:i:<freq><LF>    one per read in id order; F = the stored (canonical) strand, freq =
 *                                                           the .reads FREQ (after a restart: the count wrapped modulo 65,536)
 *   L<TAB><a><TAB><oa><TAB><b><TAB><ob><TAB><n>M<LF>        one per undirected edge, in .graph3 order: the record (a, b, type,
 *                                                           delta) with a < b (its twin gets no line); n = len(b) - delta
 * with the orientations of the edge type:
 *   type 3  fwd b prefix on fwd a suffix   + +
 *   type 2  rc b prefix on fwd a suffix    + -
 *   type 0  fwd b suffix on fwd a prefix   - -
 *   type 1  rc b suffix on fwd a prefix    - +
 * so that the last n bases of a in orientation oa equal the first n bases of b in orientation ob.  Two reads may share two
 * L lines of different types.  SAGE2GPU_ERR_STATE (with a message) before the overlap graph is built, or when the context no
 * longer holds the reads' records, lengths and frequencies; SAGE2GPU_ERR_IO when the file cannot be written. */
int sage2gpu_write_gfa(sage2gpu_ctx *ctx, const char *path);

#ifdef __cplusplus
}
#endif
#endif
