// sage2gpu -- host program: SAGE2's command line and step structure (main.cpp:11-132, 384-521) with
// steps 1-3 (organise reads, prefix/suffix hash table, economy overlap graph) running on a B200 through
// the C ABI of libsage2gpu (include/sage2gpu.h).  It writes the reference's own intermediate files
// (<prefix>.reads, <prefix>.graph3, byte for byte what `SAGE2 -s -M 3` writes), so the reference's
// steps 4-7 continue from them unchanged: `SAGE2 -m 4 -i <prefix> ...`, which this program runs
// itself when it is told where the reference binary is (--reference PATH or $SAGE2_REFERENCE_BIN).
//
// Flags are the reference's: -f/--fileInput, -l/--listInput, -k/--minOverlap, -o/--outputDir,
// -p/--prefix, -i/--inputPrefix, -m/--minStep, -M/--maxStep, -s/--saveAll, -d/--debug, -h/--help.
// Added: --device N (CUDA ordinal), --reference PATH, --gfa (the graph of step 3 also as GFA 1.0, <prefix>.gfa, formatted on
// the device: sage2gpu_write_gfa), --devices LIST (several GPUs in ONE process: one context per listed
// device; the input is dealt to the contexts piece by piece as it is read and each packs its part; every stage partitioned --
// reads organised by key range, search by id slice -- and the all-gathers between the stages done as peer copies; no NCCL,
// no Python; same files out).  The table is replicated on every context (built by key-hash shard, all-gathered) when it fits
// beside the later stages on every GPU, otherwise sharded by key hash with the window probes routed through peer-memory
// mailboxes (low-memory mode); SAGE2GPU_TABLE_LAYOUT=replicated|sharded forces the choice, the log states it.
//
// Input: plain FASTA / FASTQ text goes to the GPU in pieces and its records are split there.  BGZF files (htslib's bgzip: gzip
// members with a BC field) are inflated on the GPU as well, piece by piece of whole members, and so are ordinary gzip files
// (gzip / pigz output), piece by piece of DEFLATE blocks found on the device.  Compressed data that fails a check (CRC32,
// ISIZE, header or DEFLATE rules, truncation) stops the program with a FORMAT error naming its compressed offset.
//
// Restarts: -m 2 and -m 3 load <outputDir><inputPrefix>.reads (ReadLoader::loadReadsFromFile, readLoader.cpp:289) -- parsed
// and checked on the device, spread over the contexts with --devices -- and do not open the -f / -l inputs in steps 1-3 (the
// flags stay required, as in the reference's checkRequired).  When that file does not exist, step 1 runs from the input files.
// A file that is not exactly what saveReadsInFile writes stops the program with a FORMAT error naming the line.  <prefix>.reads is
// written when it is not the loaded file, so that `-m 4 -i <prefix>` finds it.
//
// Differences, all stated in the log: -m 3 runs as -m 2, the table is rebuilt from the reads instead of loaded from
// <prefix>.hashTable, and <prefix>.hashTable is not written (the reference's slot order is an artefact of its own
// hash function and is read by nothing but its -m 3 restart).  There is no CPU fallback: without a
// CUDA device the program stops with an error, like the reference's printError (utils.cpp:36-40).
#include <fcntl.h>
#include <getopt.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/wait.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <functional>
#include <map>
#include <mutex>
#include <sstream>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../../include/sage2gpu.h"
#include <zlib.h>

#include "fastaq.h"

namespace {

struct Options {
    int minStep = 1, maxStep = 7, minOverlap = 0, device = 0;
    bool saveAll = false, debugging = false, parseOnly = false, gfa = false;
    std::vector<int> devices;       // --devices: one context per listed GPU, every stage partitioned, peer copies between them
    std::string fileInput, listInput, outputDir, prefixName = "untitled", inputPrefix, referenceBin;
};

std::ofstream logStream;

[[noreturn]] void printError(const std::string &kind, const std::string &msg)     // utils.cpp:36-40
{
    logStream << kind << " : " << msg << "!\n";
    logStream.flush();
    std::cerr << kind << " : " << msg << "!\n";
    exit(EXIT_FAILURE);
}

std::string trim(const std::string &s)
{
    const size_t a = s.find_first_not_of(" \t\r\n"), b = s.find_last_not_of(" \t\r\n");
    return a == std::string::npos ? "" : s.substr(a, b - a + 1);
}

void printUsage()
{
    std::cout << "USAGE:\n\tsage2gpu [options] -f <inputFile> -k <minOverlap>\n\tsage2gpu [options] -l <inputList> -k <minOverlap>\n\n";
}

void printListOfArgs()
{
    std::cout << "OPTIONS (those of SAGE2):\n"
                 "\t-f|--fileInput <file>   interleaved FASTA/FASTQ file (plain or gzip; BGZF is inflated on the GPU)\n"
                 "\t-l|--listInput <file>   list of input files (f1=/f2= pairs or f= interleaved)\n"
                 "\t-k|--minOverlap <int>   minimum overlap length\n"
                 "\t-o|--outputDir <dir>    output directory\n"
                 "\t-p|--prefix <name>      prefix of the output files [untitled]\n"
                 "\t-i|--inputPrefix <name> prefix of the files a restart reads [= prefix]\n"
                 "\t-m|--minStep <1..7>     first step to run [1]; 2 and 3 load <outputDir><inputPrefix>.reads when it exists\n"
                 "\t                        (checked on the GPU; -m 3 rebuilds the hash table); without it step 1 runs\n"
                 "\t                        from the input files\n"
                 "\t-M|--maxStep <1..7>     last step to run [7]\n"
                 "\t-s|--saveAll            save the intermediate files of every step\n"
                 "\t-d|--debug\n"
                 "\t-h|--help\n"
                 "ADDED:\n"
                 "\t--device <int>          CUDA device ordinal [0]\n"
                 "\t--reference <path>      SAGE2 binary that runs steps 4-7 from the files written here\n"
                 "\t--gfa                   also write the overlap graph of step 3 as GFA 1.0: <outputDir><prefix>.gfa\n"
                 "\t                        (needs -m <= 3 and -M >= 3)\n\n";
}

// "0,1,2" or "0-3" (or a mix); a device may be listed twice (two contexts on one GPU)
std::vector<int> parseDevices(const char *arg)
{
    std::vector<int> v;
    std::stringstream ss(arg);
    std::string tok;
    while (std::getline(ss, tok, ',')) {
        const size_t dash = tok.find('-', 1);
        if (dash != std::string::npos) { for (int d = atoi(tok.substr(0, dash).c_str()); d <= atoi(tok.substr(dash + 1).c_str()); ++d) v.push_back(d); }
        else if (!tok.empty()) v.push_back(atoi(tok.c_str()));
    }
    return v;
}

void parseArgs(int argc, char **argv, Options &o)
{
    static struct option long_options[] = {
        { "help", no_argument, 0, 'h' },          { "fileInput", required_argument, 0, 'f' },
        { "minOverlap", required_argument, 0, 'k' }, { "listInput", required_argument, 0, 'l' },
        { "outputDir", required_argument, 0, 'o' }, { "prefix", required_argument, 0, 'p' },
        { "inputPrefix", required_argument, 0, 'i' }, { "minStep", required_argument, 0, 'm' },
        { "maxStep", required_argument, 0, 'M' },  { "saveAll", no_argument, 0, 's' },
        { "debug", no_argument, 0, 'd' },          { "device", required_argument, 0, 1001 },
        { "reference", required_argument, 0, 1002 }, { "parse-only", no_argument, 0, 1003 },
        { "devices", required_argument, 0, 1004 }, { "gfa", no_argument, 0, 1005 }, { 0, 0, 0, 0 } };
    bool fFlag = false, lFlag = false;
    int c, idx = 0;
    while ((c = getopt_long(argc, argv, "hf:l:k:o:p:i:m:M:sd", long_options, &idx)) != -1) {
        switch (c) {
            case 'h': std::cout << "\n"; printUsage(); printListOfArgs(); exit(0);
            case 'f': o.fileInput = optarg; fFlag = true; break;
            case 'l': o.listInput = optarg; lFlag = true; break;
            case 'k': o.minOverlap = atoi(optarg); break;
            case 'o': {
                o.outputDir = optarg;
                while (!o.outputDir.empty() && o.outputDir.back() == '/') o.outputDir.pop_back();
                if (!o.outputDir.empty() || (optarg[0] == '/')) o.outputDir += "/";
                break;
            }
            case 'p': o.prefixName = optarg; break;
            case 'i': o.inputPrefix = optarg; break;
            case 'm': o.minStep = atoi(optarg); if (o.minStep < 1) o.minStep = 1; break;
            case 'M': o.maxStep = atoi(optarg); if (o.maxStep > 7) o.maxStep = 7; break;
            case 's': o.saveAll = true; break;
            case 'd': o.debugging = true; break;
            case 1001: o.device = atoi(optarg); break;
            case 1002: o.referenceBin = optarg; break;
            case 1003: o.parseOnly = true; break;
            case 1004: o.devices = parseDevices(optarg); break;
            case 1005: o.gfa = true; break;
            case '?': std::cout << "\n"; exit(0);
            default: std::cout << "[ERROR] Wrong command line arguments!\n\n"; exit(0);
        }
    }
    if (optind < argc) {
        std::cout << "[WARNING] There are some non-option arguments: ";
        while (optind < argc) std::cout << argv[optind++] << " ";
        std::cout << "\n";
    }
    if (fFlag && lFlag) {
        std::cout << "[ERROR] Options -f|--fileInput and -l|--listInput are mutually exclusive!\n\n";
        exit(0);
    }
    if (o.referenceBin.empty() && getenv("SAGE2_REFERENCE_BIN")) o.referenceBin = getenv("SAGE2_REFERENCE_BIN");
}

bool checkRequired(Options &o)      // main.cpp:498-521
{
    bool ok = true;
    if (o.fileInput.empty() && o.listInput.empty()) {
        std::cout << "[ERROR] One of the options -f|--fileInput or -l|--listInput is required.\n";
        ok = false;
    }
    if (o.minOverlap == 0) { std::cout << "[ERROR] Option -k|--minOverlap is required.\n"; ok = false; }
    if (o.maxStep < o.minStep) { std::cout << "[ERROR] maxStep should not be smaller than minStep!\n\n"; ok = false; }
    if (o.inputPrefix.empty()) o.inputPrefix = o.prefixName;
    return ok;
}

void banner(const char *step, const char *what)
{
    const char *bar = "***********************************************************************************************************\n";
    logStream << bar << "                                               " << step << "\n" << what << "\n" << bar;
    logStream.flush();
}

// ---- step 1 input: parse on the host, upload chunk by chunk (pinned, asynchronous) -------------------
struct Chunk {
    uint8_t *bases = nullptr;
    int64_t *offsets = nullptr;
    size_t cap_bases = 0, cap_reads = 0, n_reads = 0, n_bases = 0;
    bool pinned = false;
    int owner = -1;             // context whose _append may still be reading the buffers
    uint64_t call = 0;          // number of that call (Uploader::touch)
};

// reads [first, first + count) of context `ctx`'s upload came from one stretch of a file, in file order
struct Segment {
    int ctx;
    uint64_t first, count;
};

// bytes of a text piece and of a sequential-parser chunk; SAGE2GPU_UPLOAD_PIECE_BYTES makes them smaller, so that a small
// file is spread over several contexts (tests)
size_t pieceBytes()
{
    static const size_t v = [] {
        const char *e = getenv("SAGE2GPU_UPLOAD_PIECE_BYTES");
        const long long x = e ? atoll(e) : 0;
        return x >= 4096 ? (size_t)x : (size_t)32 << 20;
    }();
    return v;
}

// One context, or several that receive the pieces of the input in turn (read ids are ranks in the sorted set, so the
// upload order is free).  The segments of the file being read say which context holds which of its records.
class Uploader {
public:
    Uploader(const std::vector<sage2gpu_ctx *> &ctx, int k) : ctx_(ctx), received_(ctx.size(), 0), last_(ctx.size(), 0)
    {
        if (ctx_.empty()) return;   // --parse-only
        for (Chunk &c : chunk_) {
            c.cap_bases = std::min<size_t>((size_t)64 << 20, 2 * pieceBytes());
            c.cap_reads = (size_t)1 << 19;
            alloc(c);
        }
        for (size_t r = 0; r < ctx_.size(); ++r)
            if (sage2gpu_load_begin(ctx_[r], k) != 0) fail((int)r);
    }
    ~Uploader()
    {
        for (Chunk &c : chunk_) release(c);
        sage2gpu_host_free(text_);
    }
    void add(const uint8_t *seq, size_t len)
    {
        Chunk *c = &chunk_[cur_];
        if (c->n_reads == c->cap_reads || c->n_bases + len > c->cap_bases) {
            flush();
            c = &chunk_[cur_];
            if (len > c->cap_bases) { release(*c); c->cap_bases = len; alloc(*c); }
        }
        memcpy(c->bases + c->n_bases, seq, len);
        c->offsets[c->n_reads] = (int64_t)c->n_bases;
        c->n_bases += len;
        c->n_reads++;
        c->offsets[c->n_reads] = (int64_t)c->n_bases;
    }
    // one context: filter, pack, sort, dedupe (organizeReads)
    void finish()
    {
        flush();
        if (sage2gpu_load_finish(ctx_[0]) != 0) fail(0);
    }
    // everything added so far is on the device after this, and no pinned buffer is in use
    void sync()
    {
        if (ctx_.empty()) return;
        flush();
        for (size_t r = 0; r < ctx_.size(); ++r) {
            if (sage2gpu_load_append(ctx_[r], nullptr, nullptr, 0) != 0) fail((int)r);
            touch((int)r);
        }
    }
    bool active() const { return !ctx_.empty(); }
    size_t contexts() const { return ctx_.size(); }
    // the context the next piece goes to
    int next() const { return next_; }
    sage2gpu_ctx *ctx(int r) const { return ctx_[r]; }
    // device record splitting of one text piece on context next(); see sage2gpu_load_append_text
    int appendText(const uint8_t *text, size_t n, bool final, int *marker, uint64_t max_records, uint64_t &consumed, uint64_t &nrec)
    {
        const int r = next_;
        const int rc = sage2gpu_load_append_text(ctx_[r], text, n, final ? 1 : 0, marker, max_records, &consumed, &nrec);
        touch(r);
        if (rc == 0 && nrec) appended(r, nrec);
        return rc;
    }
    // inflate + record splitting of one piece of BGZF members on context next(); see sage2gpu_load_append_bgzf
    int appendBgzf(const uint8_t *prefix, size_t np, const uint8_t *bgzf, size_t n, bool final, int *marker, uint64_t max_records,
                   uint64_t &consumed, uint64_t &nrec, uint8_t *rest, size_t rest_cap, uint64_t &rest_bytes, int64_t &bad_member)
    {
        const int r = next_;
        const int rc = sage2gpu_load_append_bgzf(ctx_[r], prefix, np, bgzf, n, final ? 1 : 0, marker, max_records, &consumed, &nrec, rest,
                                                 rest_cap, &rest_bytes, &bad_member);
        touch(r);
        if (rc == 0 && nrec) appended(r, nrec);
        return rc;
    }
    // inflate + record splitting of one piece of an ordinary gzip stream on context next(); see sage2gpu_load_append_gzip
    int appendGzip(const uint8_t *prefix, size_t np, const uint8_t *gz, size_t n, bool final, uint64_t text_bound, sage2gpu_gzip_state *state,
                   int *marker, uint64_t max_records, uint64_t &consumed, uint64_t &nrec, uint8_t *rest, size_t rest_cap, uint64_t &rest_bytes,
                   uint64_t &in_consumed, int64_t &bad_offset)
    {
        const int r = next_;
        const int rc = sage2gpu_load_append_gzip(ctx_[r], prefix, np, gz, n, final ? 1 : 0, text_bound, state, marker, max_records, &consumed, &nrec,
                                                 rest, rest_cap, &rest_bytes, &in_consumed, &bad_offset);
        touch(r);
        if (rc == 0 && nrec) appended(r, nrec);
        return rc;
    }
    // pinned buffer for raw file text (device-side record splitting)
    uint8_t *text(size_t &cap)
    {
        if (!text_) { text_ = (uint8_t *)sage2gpu_host_alloc(pieceBytes()); if (!text_) printError("MEM_ALLOC", "pinned text buffer"); }
        cap = pieceBytes();
        return text_;
    }
    std::vector<Segment> takeSegments() { std::vector<Segment> s; s.swap(segs_); return s; }
    // drops the records [keep, end) of a file, in file order, from the contexts that hold them
    void removeTail(const std::vector<Segment> &file, uint64_t keep)
    {
        uint64_t end = 0;
        for (const Segment &s : file) end += s.count;
        for (size_t i = file.size(); i-- > 0 && end > keep;) {     // from the back: the earlier segments of a context keep their place
            const Segment &s = file[i];
            const uint64_t start = end - s.count, from = std::max(start, keep);
            if (sage2gpu_load_remove(ctx_[s.ctx], s.first + (from - start), end - from) != 0) fail(s.ctx);
            touch(s.ctx);
            received_[s.ctx] -= end - from;
            end = start;
        }
    }
    const std::vector<uint64_t> &received() const { return received_; }
    [[noreturn]] void fail(int r) { printError("CUDA", sage2gpu_last_error(ctx_[r])); }

private:
    uint8_t *text_ = nullptr;
    void alloc(Chunk &c)
    {
        c.bases = (uint8_t *)sage2gpu_host_alloc(c.cap_bases);
        c.offsets = (int64_t *)sage2gpu_host_alloc((c.cap_reads + 1) * sizeof(int64_t));
        c.pinned = c.bases && c.offsets;
        if (!c.pinned) printError("MEM_ALLOC", "pinned upload buffers");
        c.n_reads = c.n_bases = 0;
        c.offsets[0] = 0;
    }
    void release(Chunk &c)
    {
        sage2gpu_host_free(c.bases);
        sage2gpu_host_free(c.offsets);
        c.bases = nullptr; c.offsets = nullptr;
    }
    uint64_t touch(int r) { return last_[r] = ++calls_; }
    void appended(int r, uint64_t n)
    {
        if (!segs_.empty() && segs_.back().ctx == r && segs_.back().first + segs_.back().count == received_[r]) segs_.back().count += n;
        else segs_.push_back(Segment{ r, received_[r], n });
        received_[r] += n;
        next_ = (next_ + 1) % (int)ctx_.size();
    }
    void flush()
    {
        Chunk &c = chunk_[cur_];
        if (c.n_reads) {
            // returns once the copy of that context's PREVIOUS chunk is complete; this chunk's copy runs while the parser fills
            // the other buffer
            const int r = next_;
            if (sage2gpu_load_append(ctx_[r], c.bases, c.offsets, (int64_t)c.n_reads) != 0) fail(r);
            c.owner = r;
            c.call = touch(r);
            appended(r, c.n_reads);
        }
        cur_ ^= 1;
        Chunk &n = chunk_[cur_];
        // a chunk's buffers are free once a LATER call on the context it went to has returned
        if (n.owner >= 0 && last_[n.owner] <= n.call) {
            if (sage2gpu_load_append(ctx_[n.owner], nullptr, nullptr, 0) != 0) fail(n.owner);
            touch(n.owner);
        }
        n.owner = -1;
        n.n_reads = n.n_bases = 0;
        n.offsets[0] = 0;
    }
    std::vector<sage2gpu_ctx *> ctx_;
    std::vector<uint64_t> received_, last_;     // reads per context; number of the latest call on it
    std::vector<Segment> segs_;
    Chunk chunk_[2];
    int cur_ = 0, next_ = 0;
    uint64_t calls_ = 0;
};

// --parse-only: the input side alone (no device): record count, base count and an FNV-1a checksum of the
// sequences in the order they would be uploaded.  Used by the CPU tests of the parser / list grammar.
struct ParseSink {
    uint64_t reads = 0, bases = 0, fnv = 1469598103934665603ull;
    void add(const uint8_t *s, size_t n)
    {
        for (size_t i = 0; i < n; ++i) { fnv ^= s[i]; fnv *= 1099511628211ull; }
        fnv ^= 0xFF; fnv *= 1099511628211ull;
        reads++; bases += n;
    }
};
ParseSink *g_parse_sink = nullptr;

// sequential parser (any layout the reference accepts) on `in`, at most max_records records
uint64_t parseSequential(Uploader &up, sg_host::FastAQStream &in, uint64_t max_records)
{
    std::vector<uint8_t> seq;
    uint64_t len = 0, n = 0;
    while (n < max_records) {
        seq.clear();
        if (!in.next(seq, len)) break;
        if (g_parse_sink) g_parse_sink->add(seq.data(), seq.size());
        else up.add(seq.data(), seq.size());
        ++n;
    }
    return n;
}

uint32_t le32(const uint8_t *p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }

// The gzip member header at p[0, n): its size (BSIZE + 1) when it is a BGZF member (gzip magic, FEXTRA, a `BC` subfield with
// SLEN 2); 0 when it is not; -1 when n is too short to tell
long bgzfMemberBytes(const uint8_t *p, size_t n)
{
    if (n < 12) return -1;
    if (p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) return 0;
    const size_t xlen = (size_t)p[10] | (size_t)p[11] << 8;
    if (n < 12 + xlen) return -1;
    for (size_t i = 12; i + 4 <= 12 + xlen;) {
        const size_t slen = (size_t)p[i + 2] | (size_t)p[i + 3] << 8;
        if (i + 4 + slen > 12 + xlen) break;
        if (p[i] == 'B' && p[i + 1] == 'C' && slen == 2) return 1 + (long)((size_t)p[i + 4] | (size_t)p[i + 5] << 8);
        i += 4 + slen;
    }
    return 0;
}

// the sequential parser from compressed offset `off` of the file on (a member boundary, so zlib starts a fresh stream) after the
// host text pending[0, n)
uint64_t parseRestSequential(Uploader &up, int fd, off_t off, const uint8_t *pending, size_t n, uint64_t max_records, const std::string &path)
{
    if (lseek(fd, off, SEEK_SET) != off) { close(fd); throw std::runtime_error("cannot read " + path); }
    gzFile gz = gzdopen(fd, "r");
    if (!gz) { close(fd); throw std::runtime_error("cannot read " + path); }
    gzbuffer(gz, 1 << 20);
    sg_host::FastAQStream in(gz, pending, n);           // takes the handle
    const uint64_t got = parseSequential(up, in, max_records);
    up.sync();
    return got;
}

// A BGZF file: the compressed bytes are read with read(2) into pinned memory, cut into pieces of whole members whose texts
// add up to at most pieceBytes() (at least one member), and every piece is inflated and split on the device.  The text a
// piece leaves over (at most one record) comes back to the host and goes in front of the next piece, which may go to
// another context.  Irregular text, and members without a `BC` field, continue on the sequential parser.
uint64_t readBgzf(Uploader &up, int fd, const std::string &path, uint64_t max_records, bool &used_device_parser)
{
    const size_t piece = pieceBytes(), ccap = piece + ((size_t)1 << 20), rcap = 2 * piece + ((size_t)1 << 17);
    uint8_t *cbuf = (uint8_t *)sage2gpu_host_alloc(ccap), *pre = (uint8_t *)sage2gpu_host_alloc(rcap),
            *rest = (uint8_t *)sage2gpu_host_alloc(rcap);
    if (!cbuf || !pre || !rest) printError("MEM_ALLOC", "pinned BGZF buffers");
    struct Free { uint8_t *a, *b, *c; ~Free() { sage2gpu_host_free(a); sage2gpu_host_free(b); sage2gpu_host_free(c); } } release{ cbuf, pre, rest };
    size_t have = 0, np = 0;               // compressed bytes in cbuf (from file offset base on); host text in front of the next piece
    off_t base = 0;
    bool eof = false;
    int marker = 0;
    uint64_t total = 0;
    auto fill = [&] {
        while (have < ccap && !eof) {
            const ssize_t n = read(fd, cbuf + have, ccap - have);
            if (n < 0) { close(fd); throw std::runtime_error("cannot read " + path); }
            if (n == 0) eof = true; else have += (size_t)n;
        }
    };
    auto fallback = [&](off_t off, const char *why) {
        logStream << "\tBGZF file " << path << ": " << why << " at compressed offset " << off
                  << "; the rest of the file continues on the sequential parser (host zlib).\n";
        return total + parseRestSequential(up, fd, off, pre, np, max_records - total, path);
    };
    up.sync();
    for (;;) {
        fill();
        // whole members from the front of cbuf
        size_t end = 0;
        uint64_t text = 0;
        bool plain = false;                // the next member has no BC field
        for (;;) {
            if (end == have) break;
            const long mb = bgzfMemberBytes(cbuf + end, have - end);
            if (mb == 0) { plain = true; break; }
            if (mb < 0 || end + (size_t)mb > have) {
                if (end > 0 || !eof) break;     // the rest of the member comes with the next fill
                printError("FORMAT", path + ": BGZF member at compressed offset " + std::to_string(base + (off_t)end) +
                                         (mb < 0 ? ": truncated header" : ": BSIZE reaches past the end of the file"));
            }
            if ((size_t)mb < 26) printError("FORMAT", path + ": BGZF member at compressed offset " + std::to_string(base + (off_t)end) + ": BSIZE too small");
            const uint32_t isize = le32(cbuf + end + mb - 4);
            if (end > 0 && text + isize > piece) break;
            end += (size_t)mb;
            text += isize;
        }
        if (end == 0 && plain) return fallback(base, "a gzip member without a BC field");
        const bool final = end == have && eof;
        uint64_t consumed = 0, nrec = 0, nrest = 0;
        int64_t bad = -1;
        const int r = up.next();
        const int rc = up.appendBgzf(pre, np, cbuf, end, final, &marker, max_records - total, consumed, nrec, rest, rcap, nrest, bad);
        if (rc == SAGE2GPU_ERR_FORMAT && bad >= 0) {
            // the member's offset: walk the piece's members once more
            size_t off = 0;
            for (int64_t i = 0; i < bad; ++i) off += (size_t)bgzfMemberBytes(cbuf + off, end - off);
            std::string e = sage2gpu_last_error(up.ctx(r));
            const size_t colon = e.find("): ");
            printError("FORMAT", path + ": BGZF member at compressed offset " + std::to_string(base + (off_t)off) + ": " +
                                     (colon == std::string::npos ? e : e.substr(colon + 3)));
        }
        if (rc == SAGE2GPU_ERR_FORMAT) return fallback(base, "text not in the regular 4-line FASTQ / 2-line FASTA layout");
        if (rc != 0) up.fail(r);
        used_device_parser = true;
        total += nrec;
        if (nrest > rcap) printError("MEM_ALLOC", "a record longer than the BGZF rest buffer");
        std::swap(pre, rest);
        np = (size_t)nrest;
        memmove(cbuf, cbuf + end, have - end);
        have -= end;
        base += (off_t)end;
        if (total >= max_records || final) break;
        if (consumed == 0) return fallback(base, "a record longer than a piece");
    }
    up.sync();
    close(fd);
    return total;
}

// Text bound of a gzip piece when one context reads the file.  A piece's parallelism is its number of DEFLATE blocks (one warp
// each): a 32 MB piece of level-6 FASTQ holds some 180, a warp or two per SM of a B200, so one context takes 8 pieces' worth at
// once (some 1,450 ranges, about 10 warps per SM).  Several contexts keep pieceBytes(), so that the input is spread over them.
constexpr size_t kGzipSingleContextPieces = 8;

// An ordinary gzip file (one member, or members concatenated): the compressed bytes are read with read(2) into pinned memory
// and every piece is inflated and split on the device (sage2gpu_load_append_gzip), at most pieceBytes() of text each, or
// kGzipSingleContextPieces times that with one context.  The
// piece state (block boundary, the member's last 32 KiB, running CRC and length) and the text a piece leaves over stay on the
// host and go with the next piece to whichever context takes it.  Irregular text continues on the sequential parser: zlib
// reopens the file and skips the text the device consumed.
uint64_t readGzip(Uploader &up, int fd, const std::string &path, uint64_t max_records, bool &used_device_parser)
{
    const size_t piece = pieceBytes(), rcap = 2 * piece + ((size_t)1 << 17);
    const size_t bound = up.contexts() == 1 ? kGzipSingleContextPieces * piece : piece;
    size_t ccap = bound / 4 + ((size_t)1 << 20);
    uint8_t *cbuf = (uint8_t *)sage2gpu_host_alloc(ccap), *pre = (uint8_t *)sage2gpu_host_alloc(rcap), *rest = (uint8_t *)sage2gpu_host_alloc(rcap);
    sage2gpu_gzip_state *gs = (sage2gpu_gzip_state *)calloc(1, sizeof(sage2gpu_gzip_state));
    if (!cbuf || !pre || !rest || !gs) printError("MEM_ALLOC", "pinned gzip buffers");
    struct Free {
        uint8_t **a, **b, **c;
        sage2gpu_gzip_state *s;
        ~Free() { sage2gpu_host_free(*a); sage2gpu_host_free(*b); sage2gpu_host_free(*c); free(s); }
    } release{ &cbuf, &pre, &rest, gs };
    size_t have = 0, np = 0;               // compressed bytes in cbuf (from gs->offset on); host text in front of the next piece
    size_t feed = bound / 4 + ((size_t)1 << 16);     // compressed bytes per piece, from the ratio seen so far
    bool eof = false;
    int marker = 0;
    uint64_t total = 0, text_done = 0;     // records; text bytes the device consumed
    auto fill = [&](size_t want) {
        if (want > ccap) {
            uint8_t *b = (uint8_t *)sage2gpu_host_alloc(want);
            if (!b) printError("MEM_ALLOC", "pinned gzip buffers");
            memcpy(b, cbuf, have);
            sage2gpu_host_free(cbuf);
            cbuf = b;
            ccap = want;
        }
        while (have < want && !eof) {
            const ssize_t n = read(fd, cbuf + have, want - have);
            if (n < 0) { close(fd); throw std::runtime_error("cannot read " + path); }
            if (n == 0) eof = true; else have += (size_t)n;
        }
    };
    auto fallback = [&](const char *why) {
        logStream << "\tgzip file " << path << ": " << why << " at text offset " << text_done
                  << "; the rest of the file continues on the sequential parser (host zlib).\n";
        if (lseek(fd, 0, SEEK_SET) != 0) { close(fd); throw std::runtime_error("cannot read " + path); }
        gzFile gz = gzdopen(fd, "r");
        if (!gz) { close(fd); throw std::runtime_error("cannot read " + path); }
        gzbuffer(gz, 1 << 20);
        if (gzseek(gz, (z_off_t)(text_done + np), SEEK_SET) < 0) { gzclose(gz); throw std::runtime_error("cannot read " + path); }
        sg_host::FastAQStream in(gz, pre, np);          // takes the handle
        const uint64_t got = parseSequential(up, in, max_records - total);
        up.sync();
        return total + got;
    };
    up.sync();
    for (;;) {
        fill(feed);
        const size_t take = std::min(have, feed);
        const bool final = eof && take == have;
        uint64_t consumed = 0, nrec = 0, nrest = 0, nin = 0;
        int64_t bad = -1;
        const int r = up.next();
        const int rc = up.appendGzip(pre, np, cbuf, take, final, bound, gs, &marker, max_records - total, consumed, nrec, rest, rcap, nrest, nin, bad);
        if (rc == SAGE2GPU_ERR_FORMAT && bad >= 0) {
            const std::string e = sage2gpu_last_error(up.ctx(r));
            const size_t colon = e.find(": ");
            printError("FORMAT", path + ": gzip data at compressed offset " + std::to_string(bad) + ": " +
                                     (colon == std::string::npos ? e : e.substr(colon + 2)));
        }
        if (rc == SAGE2GPU_ERR_FORMAT) return fallback("text not in the regular 4-line FASTQ / 2-line FASTA layout");
        if (rc != 0) up.fail(r);
        used_device_parser = true;
        total += nrec;
        text_done += consumed;
        if (total >= max_records) break;
        if (nrest > rcap) {                // only the start of the unfinished record came back: zlib takes it from its start
            np = 0;
            return fallback("a record longer than a piece");
        }
        const uint64_t text = consumed + nrest - np;    // inflated by this piece
        std::swap(pre, rest);
        np = (size_t)nrest;
        memmove(cbuf, cbuf + nin, have - nin);
        have -= (size_t)nin;
        if (gs->done) break;
        if (nin == 0) feed *= 2;           // no complete block in the piece
        else feed = std::max<size_t>((size_t)1 << 16, (size_t)((double)bound * nin / std::max<uint64_t>(text, 1)) + ((size_t)1 << 14));
        if (consumed == 0 && np > piece) return fallback("a record longer than a piece");
    }
    up.sync();
    close(fd);
    return total;
}

// One file: raw text goes to the device in 32 MB pieces and the records are split there
// (sage2gpu_load_append_text); text that is not in the regular layout is parsed sequentially from that point on.
// BGZF and other gzip files are inflated on the device too (readBgzf, readGzip); `inflated` names which.
uint64_t readFile(Uploader &up, const std::string &path, uint64_t max_records, bool &used_device_parser, std::string &inflated)
{
    used_device_parser = false;
    inflated.clear();
    if (!up.active()) {                    // --parse-only
        sg_host::FastAQStream in(path);
        return parseSequential(up, in, max_records);
    }
    const int fd = open(path.c_str(), O_RDONLY);
    if (fd < 0) throw std::runtime_error("cannot open " + path);
    unsigned char magic[1024] = { 0 };
    const ssize_t nm = pread(fd, magic, sizeof(magic), 0);
    if (nm >= 2 && magic[0] == 0x1f && magic[1] == 0x8b) {
        const bool bgzf = bgzfMemberBytes(magic, (size_t)nm) > 0;
        const uint64_t n = bgzf ? readBgzf(up, fd, path, max_records, used_device_parser) : readGzip(up, fd, path, max_records, used_device_parser);
        if (used_device_parser) inflated = bgzf ? "BGZF" : "gzip";
        return n;
    }
    // plain text is read with read(2) straight into the pinned buffer
    size_t cap = 0, have = 0;
    uint8_t *buf = up.text(cap);
    int marker = 0;                        // the file's record layout ('@' / '>'), found in its first piece; the same for every context
    bool eof = false;
    uint64_t total = 0;
    up.sync();                             // the records of this file form segments of their own
    for (;;) {
        while (have < cap && !eof) {
            const long n = (long)read(fd, buf + have, cap - have);
            if (n <= 0) eof = true; else have += (size_t)n;
        }
        if (have == 0) break;
        uint64_t consumed = 0, nrec = 0;
        const int r = up.next();
        const int rc = up.appendText(buf, have, eof, &marker, max_records - total, consumed, nrec);
        if (rc == SAGE2GPU_ERR_FORMAT || (rc == 0 && consumed == 0 && !eof)) {
            gzFile gz = gzdopen(fd, "r");                     // transparent mode, continues at the descriptor's offset
            if (!gz) { close(fd); throw std::runtime_error("cannot read " + path); }
            sg_host::FastAQStream in(gz, buf, have);          // takes the handle; continues behind what the device consumed
            total += parseSequential(up, in, max_records - total);
            up.sync();
            return total;
        }
        if (rc != 0) up.fail(r);
        used_device_parser = true;
        total += nrec;
        have -= (size_t)consumed;
        if (have) memmove(buf, buf + consumed, have);
        if (total >= max_records || (eof && have == 0)) break;
    }
    close(fd);
    return total;
}

uint64_t readDataset(Uploader &up, const std::string &f1, const std::string &f2)      // readLoader.cpp:133-174
{
    logStream << "In function readDatasetInBytes().\n";
    logStream << "Reading from file: " << f1 << " " << (f2.empty() ? "" : "& " + f2) << "\n";
    logStream.flush();
    uint64_t n = 0;
    try {
        bool dev1 = false, dev2 = false;
        std::string inf1, inf2;
        if (f2.empty()) {
            n = readFile(up, f1, UINT64_MAX, dev1, inf1);
            up.takeSegments();
        } else if (!up.active()) {
            sg_host::MatePairStream in(f1, f2);     // --parse-only keeps the reference's alternating order
            std::vector<uint8_t> seq;
            uint64_t len = 0;
            for (;;) { seq.clear(); if (!in.next(seq, len)) break; g_parse_sink->add(seq.data(), seq.size()); ++n; }
        } else {
            // The reference alternates mate 1 / mate 2 and stops when a file ends (inputReader.cpp:26-49): with n1 and n2
            // records it keeps min(n1, n2 + 1) of file 1 and min(n2, n1) of file 2.  Read ids are ranks in the sorted set,
            // so the upload order is free: file 1, then file 2 capped at n1, then the surplus of file 1 (its last records, in
            // whichever contexts they went to) is dropped.
            const uint64_t n1 = readFile(up, f1, UINT64_MAX, dev1, inf1);
            const std::vector<Segment> file1 = up.takeSegments();
            const uint64_t n2 = readFile(up, f2, n1, dev2, inf2);
            up.takeSegments();
            uint64_t keep1 = n1;
            if (n1 > n2 + 1) {
                keep1 = n2 + 1;
                up.removeTail(file1, keep1);
            }
            n = keep1 + n2;
        }
        logStream << "\tRecords split on the device: " << ((dev1 || dev2) ? "yes" : "no (sequential parser)")
                  << (inf1.empty() && inf2.empty() ? "" : "; " + (inf1.empty() ? inf2 : inf2.empty() || inf2 == inf1 ? inf1 : inf1 + " and " + inf2) +
                                                             " text inflated on the device")
                  << "\n";
    } catch (const std::runtime_error &e) {
        printError("OPEN_FILE", e.what());
    }
    logStream << "\t" << std::setw(21) << "Total reads in file: " << n << "\n";
    logStream.flush();
    return n;
}

uint64_t loadFromList(Uploader &up, const std::string &listPath)      // readLoader.cpp:73-131
{
    std::ifstream fin(listPath.c_str());
    if (!fin.is_open()) printError("OPEN_FILE", listPath);
    std::string line, val1;
    uint32_t mateFile = 0;
    uint64_t total = 0;
    while (std::getline(fin, line)) {
        if (line.empty() || line[0] == '#') continue;
        const size_t pos = line.find('=');
        if (pos == std::string::npos) { std::cout << "[ERROR] List of input files in a wrong format!\n\n"; exit(0); }
        const std::string var = trim(line.substr(0, pos)), val = trim(line.substr(pos + 1));
        if (mateFile % 2 == 0 && var == "f1") val1 = val;
        else if (mateFile % 2 == 0 && var == "f") { total += readDataset(up, val, ""); mateFile++; }
        else if (mateFile % 2 == 1 && var == "f2") total += readDataset(up, val1, val);
        else { std::cout << "[ERROR] List of input files in a wrong format!\n\n"; exit(0); }
        mateFile++;
    }
    logStream << std::setw(20) << "Number of datasets: " << mateFile / 2 << "\n";
    return total;
}

double seconds_since(const std::chrono::steady_clock::time_point &t0)
{
    return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}

// --gfa: <prefix>.gfa from a context that holds the reads and the complete edge list
void saveGfa(sage2gpu_ctx *ctx, const std::string &base)
{
    auto t = std::chrono::steady_clock::now();
    if (const int rc = sage2gpu_write_gfa(ctx, (base + ".gfa").c_str())) printError(rc == SAGE2GPU_ERR_IO ? "OPEN_FILE" : "CUDA", sage2gpu_last_error(ctx));
    logStream << "Function saveGfa in " << seconds_since(t) << " sec.\n";
}

int runReference(const Options &o, int fromStep)
{
    std::vector<std::string> a = { o.referenceBin };
    if (!o.listInput.empty()) { a.push_back("-l"); a.push_back(o.listInput); } else { a.push_back("-f"); a.push_back(o.fileInput); }
    a.push_back("-k"); a.push_back(std::to_string(o.minOverlap));
    if (!o.outputDir.empty()) { a.push_back("-o"); a.push_back(o.outputDir); }
    a.push_back("-p"); a.push_back(o.prefixName);
    a.push_back("-i"); a.push_back(fromStep == 4 && o.minStep <= 3 ? o.prefixName : o.inputPrefix);
    a.push_back("-m"); a.push_back(std::to_string(fromStep));
    a.push_back("-M"); a.push_back(std::to_string(o.maxStep));
    if (o.saveAll) a.push_back("-s");
    std::vector<char *> argv;
    for (auto &s : a) argv.push_back(const_cast<char *>(s.c_str()));
    argv.push_back(nullptr);
    const pid_t pid = fork();
    if (pid < 0) return -1;
    if (pid == 0) { execv(argv[0], argv.data()); _exit(127); }
    int status = 0;
    waitpid(pid, &status, 0);
    return WIFEXITED(status) ? WEXITSTATUS(status) : -1;
}

}  // namespace

// ---- several GPUs in one process ---------------------------------------------------------------------------------
// One context per listed device, one host thread per context (the library calls block), peer copies between the stages.
// The input is spread over the contexts as it is read; the steps are those of sage2_b200/multi.py::partitioned_slice_steps
// (table replicated) or partitioned_slice_sharded_steps (table sharded, low-memory mode), whichever fits.
struct MultiGpu {
    std::vector<sage2gpu_ctx *> ctx;
    std::vector<int> device;
    int G() const { return (int)ctx.size(); }
    void each(const std::function<void(int)> &fn)
    {
        std::vector<std::thread> th;
        for (int r = 0; r < G(); ++r) th.emplace_back(fn, r);
        for (auto &t : th) t.join();
    }
    void check(int r, int rc) { if (rc != 0) printError("CUDA", std::string("device context ") + std::to_string(r) + ": " + sage2gpu_last_error(ctx[r])); }
    // all-gather of blocks: block q (bytes[q] bytes at byte offset off[q]) of every context's array comes from context q
    void gather(const std::vector<void *> &ptr, const std::vector<uint64_t> &off, const std::vector<uint64_t> &bytes)
    {
        each([&](int r) {
            for (int q = 0; q < G(); ++q)
                if (q != r && bytes[q]) check(r, sage2gpu_peer_copy(ctx[r], (char *)ptr[r] + off[q], ctx[q], (const char *)ptr[q] + off[q], bytes[q]));
        });
    }
};

// Rendezvous of the G threads of one sharded build: every thread passes its value and gets the maximum over all of them.
class HostSync {
public:
    explicit HostSync(int n) : n_(n) {}
    uint64_t max(uint64_t v)
    {
        std::unique_lock<std::mutex> lk(mu_);
        const uint64_t gen = gen_;
        acc_ = std::max(acc_, v);
        if (++arrived_ == n_) { result_ = acc_; acc_ = 0; arrived_ = 0; ++gen_; cv_.notify_all(); }
        else cv_.wait(lk, [&] { return gen_ != gen; });
        return result_;
    }
    void wait() { max(0); }

private:
    std::mutex mu_;
    std::condition_variable cv_;
    const int n_;
    int arrived_ = 0;
    uint64_t gen_ = 0, acc_ = 0, result_ = 0;
};

// Reads per routed batch of the sharded table (as tools/run_cfg5.py); SAGE2GPU_ROUTE_BATCH_READS makes it smaller (tests).
uint64_t routeBatchReads()
{
    const char *e = getenv("SAGE2GPU_ROUTE_BATCH_READS");
    const long long v = e ? atoll(e) : 0;
    return v > 0 ? (uint64_t)v : (uint64_t)1 << 18;
}

// Memory the stages after the table need beside it, per unique read of a context: phase-A arrays, phase-B records and
// workspace.  From the per-GPU sizes of config #5 (DESIGN.md section 4c): at full size 20 + 17.6 + 25 GB for 562 M unique
// reads (111 B per read); at half size the replicated peak of 99.8 GB less the reads (F + RC, 36 GB) and the table
// (15 GB) leaves 49 GB for 281 M unique reads (174 B per read).  Rounded up; how close it comes has not been measured.
constexpr uint64_t kReserveBytesPerUniqueRead = 192;

// One thread of the sharded build (multi.py::sharded_graph_steps over peer-memory mailboxes).  Every library call returns
// with its stream drained, so the rendezvous of the threads (HostSync) separates the steps of a routed batch; the device
// barrier (sage2gpu_mailbox_barrier) is for ranks in different processes.  Inside one process it could stall: its kernel
// spins on the device until the peers arrive, and a synchronous free of another context on the same GPU waits for it.
void shardedSteps(MultiGpu &m, HostSync &hs, std::vector<void *> &box, int r, uint64_t batch, uint64_t &redo_max, uint64_t &list_max)
{
    const int G = m.G();
    uint64_t box_reads = 0;
    auto openMailboxes = [&](uint64_t reads) {
        hs.wait();                  // nobody stores into the old mailboxes any more
        m.check(r, sage2gpu_mailbox_create(m.ctx[r], r, G, reads, nullptr, &box[r]));
        hs.wait();
        for (int q = 0; q < G; ++q) if (q != r) m.check(r, sage2gpu_mailbox_open(m.ctx[r], q, nullptr, box[q]));
        hs.wait();
        box_reads = reads;
    };
    auto route = [&](int what, uint64_t first, uint64_t count, int exact, bool posted) {
        if (!posted) m.check(r, sage2gpu_route_post(m.ctx[r], what, first, count, exact, nullptr, nullptr));
        hs.wait();
        m.check(r, sage2gpu_answer_post(m.ctx[r], exact, nullptr));
        hs.wait();
        m.check(r, sage2gpu_route_collect(m.ctx[r]));
    };
    // a list batch (redo reads, reads left for phase C) travels as ONE batch: the mailboxes of all contexts grow to the largest list
    auto fitMailbox = [&](uint64_t n_list) {
        const uint64_t need = hs.max(n_list);
        if (need > box_reads) openMailboxes(need);
        return need;
    };

    sage2gpu_counters c;
    sage2gpu_get_counters(m.ctx[r], &c);
    const uint64_t U = c.unique_reads, chunk = U ? (U + G - 1) / G : 0;
    m.check(r, sage2gpu_build_hash_table_shard(m.ctx[r], r, G));
    openMailboxes(std::max<uint64_t>(1, std::min(batch, chunk)));      // no batch is larger than a context's slice
    uint64_t first = 0, count = 0;
    m.check(r, sage2gpu_phase_a_sharded_begin(m.ctx[r], r, G, &first, &count));
    const uint64_t n_batches = chunk ? (chunk + batch - 1) / batch : 0;      // the same on every context: the steps stay in lockstep
    uint64_t redo = 0;
    for (uint64_t b = 0; b < n_batches; ++b) {
        const uint64_t lo = std::min(first + b * batch, first + count), n = std::min(batch, first + count - lo);
        route(0, lo, n, 0, false);
        uint64_t nr = 0;
        m.check(r, sage2gpu_phase_a_routed(m.ctx[r], &nr));
        redo += nr;
    }
    const uint64_t redo_all = hs.max(redo);
    if (redo_all) {
        // 24-bit tag collisions: those reads once more, with probes the owners verify
        fitMailbox(redo);
        route(2, 0, 0, 1, false);
        uint64_t left = 0;
        m.check(r, sage2gpu_phase_a_routed(m.ctx[r], &left));
        if (left) printError("CUDA", "device context " + std::to_string(r) + ": " + std::to_string(left) + " reads still unresolved after the verified pass");
    }
    m.check(r, sage2gpu_phase_a_sharded_end(m.ctx[r]));
    hs.wait();
    for (int q = 0; q < G; ++q) if (q != r) m.check(r, sage2gpu_phase_a_import(m.ctx[r], m.ctx[q], q));
    hs.wait();
    m.check(r, sage2gpu_phase_b(m.ctx[r]));
    sage2gpu_get_counters(m.ctx[r], &c);
    const uint64_t list = fitMailbox(c.left_to_explore);
    uint64_t n_list = 0;
    m.check(r, sage2gpu_route_post(m.ctx[r], 1, 0, 0, 1, &n_list, nullptr));      // reads left for phase C: the same list everywhere
    if (n_list) route(1, 0, 0, 1, true);
    m.check(r, sage2gpu_finish_graph(m.ctx[r]));
    if (r == 0) { redo_max = redo_all; list_max = list; }
}

// step 1 after the upload spread over the contexts: every context packs its part, the parts are all-gathered and every
// context organises its key range.  Returns the unique reads of every context's run.
std::vector<uint64_t> organizePartitioned(MultiGpu &m)
{
    const int G = m.G();
    // the contexts agree on the longest read: it fixes the record stride of every slice
    std::vector<int> ml(G, 0);
    m.each([&](int r) { m.check(r, sage2gpu_load_max_length(m.ctx[r], &ml[r])); });
    const int max_len = std::max(1, *std::max_element(ml.begin(), ml.end()));
    std::vector<uint64_t> counts(G, 0), good(G, 0), bp(G, 0), sw(G, 0);
    m.each([&](int r) { m.check(r, sage2gpu_load_finish_slice(m.ctx[r], max_len, &counts[r], &good[r], &bp[r], &sw[r])); });
    uint64_t N = 0, good_all = 0, bp_all = 0;
    for (int r = 0; r < G; ++r) { N += counts[r]; good_all += good[r]; bp_all += bp[r]; }
    const uint64_t SW = sw[0];
    std::vector<void *> p(G, nullptr);
    m.each([&](int r) { m.check(r, sage2gpu_raw_gather_layout(m.ctx[r], r, G, counts.data(), &p[r], nullptr, nullptr)); });
    {
        std::vector<uint64_t> off(G, 0), bytes(G, 0);
        uint64_t acc = 0;
        for (int q = 0; q < G; ++q) { off[q] = acc * SW * 8; bytes[q] = counts[q] * SW * 8; acc += counts[q]; }
        m.gather(p, off, bytes);
    }
    std::vector<uint64_t> uloc(G, 0);
    m.each([&](int r) {
        m.check(r, sage2gpu_raw_gather_finish(m.ctx[r], N, good_all, bp_all));
        m.check(r, sage2gpu_organize_partition(m.ctx[r], r, G, &uloc[r]));
    });
    return uloc;
}

// FORMAT error of a saved .reads file (utils.cpp:36-40: log, exit); `msg` names the line and the rule
[[noreturn]] void savedReadsError(const std::string &path, const std::string &msg) { printError("FORMAT", path + ", " + msg); }

// step 1 of a restart over the contexts (ReadLoader::loadReadsFromFile): context r parses the lines that start in the r-th of G
// equal byte ranges of the file's body, in its own thread; the contexts agree on the longest read and pack their lines as their
// unique runs.  Returns the lines of every context; U = the number of reads the file declares, good / bp = the sums of the slices.
std::vector<uint64_t> loadSavedPartitioned(MultiGpu &m, const std::string &path, int k, uint64_t &U, uint64_t &good, uint64_t &bp)
{
    const int G = m.G();
    uint64_t body = 0;
    if (const int rc = sage2gpu_saved_reads_info(m.ctx[0], path.c_str(), &U, &body)) {
        if (rc == SAGE2GPU_ERR_FORMAT) savedReadsError(path, sage2gpu_last_error(m.ctx[0]));
        printError("OPEN_FILE", sage2gpu_last_error(m.ctx[0]));
    }
    std::vector<uint64_t> lines(G, 0), bad(G, 0);
    std::vector<int> ml(G, 0), rc(G, 0);
    m.each([&](int r) {
        rc[r] = sage2gpu_saved_reads_slice(m.ctx[r], path.c_str(), k, body * r / G, body * (r + 1) / G, &lines[r], &ml[r], &bad[r]);
    });
    uint64_t before = 1;        // line 1 holds the number of reads
    for (int r = 0; r < G; ++r) {
        if (rc[r] == SAGE2GPU_ERR_FORMAT) {       // the first broken line: the slices before this one were parsed completely
            const std::string e = sage2gpu_last_error(m.ctx[r]);
            savedReadsError(path, "line " + std::to_string(before + bad[r]) + e.substr(e.find(": ")));
        }
        if (rc[r] == SAGE2GPU_ERR_IO) printError("OPEN_FILE", sage2gpu_last_error(m.ctx[r]));
        m.check(r, rc[r]);
        before += lines[r];
    }
    const int max_len = *std::max_element(ml.begin(), ml.end());
    std::vector<uint64_t> uloc(G, 0), g(G, 0), b(G, 0);
    m.each([&](int r) { m.check(r, sage2gpu_saved_reads_pack(m.ctx[r], r, G, std::max(1, max_len), &uloc[r], &g[r], &b[r])); });
    good = bp = 0;
    for (int r = 0; r < G; ++r) { good += g[r]; bp += b[r]; }
    return uloc;
}

// every context's unique run all-gathered: the complete reads in every context
void gatherReads(MultiGpu &m, const std::vector<uint64_t> &uloc)
{
    const int G = m.G();
    std::vector<void *> p(G, nullptr), p2(G, nullptr), p3(G, nullptr);
    std::vector<uint64_t> stride(G, 0);
    m.each([&](int r) { m.check(r, sage2gpu_reads_gather_layout(m.ctx[r], uloc.data(), &p[r], &p2[r], &p3[r], nullptr, nullptr, &stride[r])); });
    {
        std::vector<uint64_t> off(G, 0), bytes(G, 0), off2(G, 0), bytes2(G, 0);
        uint64_t acc = 0;
        for (int q = 0; q < G; ++q) { off[q] = acc * stride[0] * 8; bytes[q] = uloc[q] * stride[0] * 8; off2[q] = acc * 2; bytes2[q] = uloc[q] * 2; acc += uloc[q]; }
        m.gather(p, off, bytes);
        m.gather(p2, off2, bytes2);
        m.gather(p3, off2, bytes2);
    }
    m.each([&](int r) { m.check(r, sage2gpu_reads_gather_finish(m.ctx[r])); });
}

// steps 2 and 3 with the complete reads in every context; the result is complete in every context.  Returns whether the
// table was replicated (else every context holds one shard of it).
bool graphPartitioned(MultiGpu &m)
{
    const int G = m.G();
    std::vector<void *> p(G, nullptr), p2(G, nullptr);
    // the layout: the table replicated on every context (faster) when it fits beside the later stages on every GPU, else sharded
    sage2gpu_counters c0;
    sage2gpu_get_counters(m.ctx[0], &c0);
    std::map<int, uint64_t> need, avail;
    uint64_t rs = 0, re = 0, ss = 0, se = 0;
    for (int r = 0; r < G; ++r) {
        uint64_t fr = 0;
        m.check(r, sage2gpu_table_bytes(m.ctx[r], G, &rs, &re, &ss, &se, &fr));
        need[m.device[r]] += rs + re + kReserveBytesPerUniqueRead * c0.unique_reads;
        avail[m.device[r]] = fr;
    }
    bool replicated = true;
    for (const auto &d : need) replicated = replicated && d.second <= avail[d.first];
    const char *forced = getenv("SAGE2GPU_TABLE_LAYOUT");
    if (forced && strcmp(forced, "replicated") && strcmp(forced, "sharded")) printError("ARGUMENT", "SAGE2GPU_TABLE_LAYOUT must be replicated or sharded");
    const bool fits = replicated;
    if (forced) replicated = !strcmp(forced, "replicated");
    logStream << "Table layout: " << (replicated ? "replicated" : "sharded") << (forced ? " (SAGE2GPU_TABLE_LAYOUT)" : "") << ". Per context: replicated table "
              << rs + re << " bytes (slots " << rs << ", entries <= " << re << "), sharded table " << ss + se << " bytes (slots " << ss
              << ", entries <= " << se << "), reserve for the later stages " << kReserveBytesPerUniqueRead * c0.unique_reads << " bytes ("
              << kReserveBytesPerUniqueRead << " per unique read).\n";
    for (const auto &d : need)
        logStream << "\tGPU " << d.first << ": replicated table + reserve of its contexts " << d.second << " bytes, free " << avail[d.first] << " bytes: "
                  << (d.second <= avail[d.first] ? "fits" : "does not fit") << "\n";
    logStream << "\tThe replicated table " << (fits ? "fits" : "does not fit") << " on every GPU.\n";
    logStream.flush();

    if (!replicated) {
        HostSync hs(G);
        std::vector<void *> box(G, nullptr);
        const uint64_t batch = routeBatchReads();
        uint64_t redo = 0, list = 0;
        m.each([&](int r) {
            m.check(r, sage2gpu_set_option(m.ctx[r], "low_memory", 1));
            shardedSteps(m, hs, box, r, batch, redo, list);
        });
        logStream << "\tSharded table: " << G << " shards, routed batches of " << batch << " reads; reads of the verified redo pass (max over the contexts): "
                  << redo << "; list batch of the reads left for phase C: " << list << " reads\n";
        return false;
    }
    std::vector<uint64_t> ec(G, 0), dk(G, 0), ov(G, 0), sps(G, 0);
    m.each([&](int r) {
        m.check(r, sage2gpu_build_hash_table_part(m.ctx[r], r, G));
        m.check(r, sage2gpu_table_shard_info(m.ctx[r], nullptr, &ec[r], &dk[r], &ov[r]));
    });
    m.each([&](int r) { m.check(r, sage2gpu_table_gather_layout(m.ctx[r], ec.data(), &p[r], &p2[r], &sps[r], nullptr)); });
    {
        std::vector<uint64_t> off(G, 0), bytes(G, 0), off2(G, 0), bytes2(G, 0);
        uint64_t acc = 0;
        for (int q = 0; q < G; ++q) { off[q] = (uint64_t)q * sps[0] * 8; bytes[q] = sps[0] * 8; off2[q] = acc * 4; bytes2[q] = ec[q] * 4; acc += ec[q]; }
        m.gather(p, off, bytes);
        m.gather(p2, off2, bytes2);
    }
    m.each([&](int r) {
        m.check(r, sage2gpu_table_gather_finish(m.ctx[r], ec.data(), dk.data(), ov.data()));
        m.check(r, sage2gpu_phase_a_partition(m.ctx[r], r, G));
    });
    m.each([&](int r) {
        for (int q = 0; q < G; ++q) if (q != r) m.check(r, sage2gpu_phase_a_import(m.ctx[r], m.ctx[q], q));
    });
    m.each([&](int r) { m.check(r, sage2gpu_finish_graph(m.ctx[r])); });
    return true;
}

// -m 2 / -m 3: the file a restart loads, <outputDir><inputPrefix>.reads (ReadLoader::loadReadsFromFile, readLoader.cpp:289)
std::string savedReadsPath(const Options &o) { return o.outputDir + o.inputPrefix + ".reads"; }

// the restart loads that file when it exists; otherwise step 1 runs from the input files
bool restartFromSavedReads(const Options &o) { return o.minStep >= 2 && o.minStep <= 3 && access(savedReadsPath(o).c_str(), F_OK) == 0; }

// <prefix>.reads of a restart: written (from the device, byte-identical to the loaded file) unless it IS the loaded file
bool writeReadsAfterRestart(const Options &o, const std::string &base)
{
    if (base + ".reads" != savedReadsPath(o)) return true;
    logStream << "NOTE: " << base << ".reads is the file this restart loaded: not rewritten.\n";
    return false;
}

// --devices with more than one entry: steps 1-3 partitioned over the listed GPUs, the same files and log lines out
int runOnSeveralDevices(const Options &o, const std::string &base)
{
    MultiGpu m;
    for (int d : o.devices) {
        sage2gpu_ctx *c = nullptr;
        if (sage2gpu_create(&c, d) != 0) printError("CUDA", "no usable CUDA device " + std::to_string(d) + " (libsage2gpu has no CPU fallback)");
        m.ctx.push_back(c);
        m.device.push_back(d);
    }
    logStream << "Devices: " << m.G() << " contexts (one per listed GPU), the input spread over them, every stage partitioned, peer copies between the stages.\n";
    const bool restart = restartFromSavedReads(o);
    auto t0 = std::chrono::steady_clock::now();
    std::vector<uint64_t> uloc;
    uint64_t declared = 0, good = 0, bp = 0;
    if (restart) {
        banner("STEP 1", "                                     loading reads from file");
        uloc = loadSavedPartitioned(m, savedReadsPath(o), o.minOverlap, declared, good, bp);
        logStream << "\tLines parsed per context:";
        for (uint64_t n : uloc) logStream << " " << n;
        logStream << "\n";
    } else {
        banner("STEP 1", "                                          organizing reads");
        Uploader up(m.ctx, o.minOverlap);
        if (!o.listInput.empty()) loadFromList(up, o.listInput);
        else readDataset(up, o.fileInput, "");
        up.sync();
        logStream << "Parsed and uploaded in " << seconds_since(t0) << " sec.\n";
        logStream << "\tReads received per context:";
        for (uint64_t n : up.received()) logStream << " " << n;
        logStream << "\n";
    }
    banner("STEPS 2-3", "                             building hash table and overlap graph");
    auto t1 = std::chrono::steady_clock::now();
    if (!restart) uloc = organizePartitioned(m);
    gatherReads(m, uloc);
    if (restart) {      // the count and the order of the complete reads (pairs across two slices too), then the counters
        std::vector<uint64_t> bad(m.G(), 0);
        std::vector<int> rc(m.G(), 0);
        m.each([&](int r) { rc[r] = sage2gpu_saved_reads_finish(m.ctx[r], declared, good, bp, &bad[r]); });
        for (int r = 0; r < m.G(); ++r) {
            if (rc[r] == SAGE2GPU_ERR_FORMAT) savedReadsError(savedReadsPath(o), sage2gpu_last_error(m.ctx[r]));
            m.check(r, rc[r]);
        }
        logStream << "Function loadReadsFromFile() on " << m.G() << " devices in " << seconds_since(t0) << " sec.\n";
    }
    const bool replicated = graphPartitioned(m);
    logStream << "Functions organizeReads() .. sortEconomyGraph() on " << m.G() << " devices in " << seconds_since(t1) << " sec.\n";
    sage2gpu_counters cnt;
    sage2gpu_get_counters(m.ctx[0], &cnt);
    if (!replicated) {      // one shard per context: the table is the sum of the shards
        cnt.table_capacity = cnt.distinct_keys = cnt.keys_over_threshold = 0;
        for (sage2gpu_ctx *c : m.ctx) {
            sage2gpu_counters s;
            sage2gpu_get_counters(c, &s);
            cnt.table_capacity += s.table_capacity; cnt.distinct_keys += s.distinct_keys; cnt.keys_over_threshold += s.keys_over_threshold;
        }
    }
    logStream << std::setw(20) << "Total reads: " << cnt.total_reads << "\n";
    logStream << std::setw(20) << "Good reads: " << cnt.good_reads << "\n";
    logStream << std::setw(20) << "Bad reads: " << cnt.total_reads - cnt.good_reads << "\n";
    logStream << "\t" << std::setw(21) << "Average read length: " << cnt.avg_len << "\n";
    logStream << "\tNumber of unique reads: " << cnt.unique_reads << "\n";
    logStream << "\tSize of hash table: " << cnt.table_capacity << " slots, " << cnt.distinct_keys << " distinct keys"
              << (replicated ? "" : " (sum over the shards)") << "\n";
    logStream << "\tNumber of hashes over threshold: " << cnt.keys_over_threshold << "\n";
    logStream << "\tTotal reads contained by extension: " << cnt.contained_ext << "\n";
    logStream << "\tTotal reads contained by size: " << cnt.contained_size << "\n";
    logStream << "\tTotal reads left to explore: " << cnt.left_to_explore << "\n";
    logStream << "\tTotal edges inserted: " << cnt.edges_inserted_c << "\n";
    logStream << "\tTotal transitive edges removed: " << cnt.transitive_removed << "\n";
    logStream << "\tEdges in the overlap graph: " << cnt.n_edges << "\n";
    if ((!restart || writeReadsAfterRestart(o, base)) && sage2gpu_write_reads(m.ctx[0], (base + ".reads").c_str()) != 0)
        printError("OPEN_FILE", sage2gpu_last_error(m.ctx[0]));
    // the graph from the LAST context: every context must hold the complete result
    if (sage2gpu_write_graph3(m.ctx[m.G() - 1], (base + ".graph3").c_str()) != 0) printError("OPEN_FILE", sage2gpu_last_error(m.ctx[m.G() - 1]));
    // the GFA needs the reads and the complete edge list in one context: ctx[0], which wrote .reads.  Both layouts leave them in
    // every context -- gatherReads gives each the complete reads, finish_graph the complete edges -- and the low-memory mode of
    // the sharded layout releases only the packed input, the unique runs before the gather, the table and the workspace
    if (o.gfa) saveGfa(m.ctx[0], base);
    logStream.flush();
    for (sage2gpu_ctx *c : m.ctx) sage2gpu_destroy(c);
    if (o.maxStep <= 3) return 0;
    if (o.referenceBin.empty()) {
        std::cout << "sage2gpu: steps 1-3 done (" << base << ".reads, " << base << ".graph3); continue with SAGE2 -m 4 -i " << o.prefixName << "\n";
        return 0;
    }
    logStream << "Running " << o.referenceBin << " -m 4 for steps 4-" << o.maxStep << ".\n";
    logStream.close();
    return runReference(o, 4);
}

int main(int argc, char **argv)
{
    Options o;
    parseArgs(argc, argv, o);
    if (!checkRequired(o)) {
        std::cout << "\n";
        printUsage();
        std::cout << "(For more information run ./sage2gpu -h)\n\n";
        exit(0);
    }
    if (o.gfa && (o.minStep > 3 || o.maxStep < 3)) {     // the graph of step 3 is what --gfa writes: refused before any work
        std::cerr << "[ERROR] --gfa writes the overlap graph of step 3: it needs -m <= 3 and -M >= 3 (given -m " << o.minStep << " -M "
                  << o.maxStep << ")\n";
        return 1;
    }
    if (!o.outputDir.empty()) {
        const std::string cmd = "mkdir -p '" + o.outputDir + "'";
        if (system(cmd.c_str()) != 0) std::cerr << "[WARNING] cannot create " << o.outputDir << "\n";
    }
    if (o.parseOnly) {
        ParseSink sink;
        g_parse_sink = &sink;
        logStream.open("/dev/null");
        Uploader none({}, o.minOverlap);
        if (!o.listInput.empty()) loadFromList(none, o.listInput);
        else readDataset(none, o.fileInput, "");
        printf("{\"reads\": %llu, \"bases\": %llu, \"fnv1a\": \"%016llx\"}\n", (unsigned long long)sink.reads,
               (unsigned long long)sink.bases, (unsigned long long)sink.fnv);
        return 0;
    }
    if (o.minStep >= 4) {       // nothing of ours to do: the reference's own steps
        if (o.referenceBin.empty()) { std::cerr << "[ERROR] steps 4-7 are the reference's: give --reference <SAGE2 binary>\n"; return 1; }
        return runReference(o, o.minStep);
    }

    const std::string base = o.outputDir + o.prefixName;
    logStream.open((base + (o.maxStep > 3 ? ".gpu.log" : ".log")).c_str());     // SAGE2 -m 4 rewrites <prefix>.log
    logStream << std::fixed << std::setprecision(2);
    logStream << "***********************************************************************************************************\n";
    logStream << "\tEXECUTING PROGRAM: sage2gpu (SAGE2 steps 1-3 on libsage2gpu)\n";
    if (!o.listInput.empty()) logStream << "\t  INPUT LIST PATH: " << o.listInput << "\n";
    else logStream << "\t  INPUT FILE PATH: " << o.fileInput << "\n";
    logStream << "\t OUTPUT DIRECTORY: " << o.outputDir << "\n";
    logStream << "\t    OUTPUT PREFIX: " << o.prefixName << "\n";
    logStream << "\t  MINIMUM OVERLAP: " << o.minOverlap << "\n";
    logStream << "\t       START STEP: " << o.minStep << "\n";
    logStream << "\t         END STEP: " << o.maxStep << "\n";
    logStream << "\t   SAVE ALL FILES: " << (o.saveAll ? "TRUE" : "FALSE") << "\n";
    logStream << "***********************************************************************************************************\n\n";
    const bool restart = restartFromSavedReads(o);
    if (restart) {
        logStream << "Restart at step " << o.minStep << ": the reads are loaded from " << savedReadsPath(o)
                  << " (ReadLoader::loadReadsFromFile); the input files are not read.\n";
        if (o.minStep == 3)
            logStream << "NOTE: -m 3 runs as -m 2: the hash table is rebuilt from the reads (" << o.inputPrefix << ".hashTable is not read).\n";
    } else if (o.minStep > 1) {
        logStream << "NOTE: " << savedReadsPath(o) << " does not exist: -m " << o.minStep << " runs step 1 from the input files (same result).\n";
    }
    logStream.flush();

    if (o.devices.size() > 1) return runOnSeveralDevices(o, base);
    if (o.devices.size() == 1) o.device = o.devices[0];
    sage2gpu_ctx *ctx = nullptr;
    if (sage2gpu_create(&ctx, o.device) != 0)
        printError("CUDA", "no usable CUDA device " + std::to_string(o.device) + " (libsage2gpu has no CPU fallback)");
    sage2gpu_counters cnt;

    // ---- step 1 -------------------------------------------------------------------------------------
    auto t0 = std::chrono::steady_clock::now();
    if (restart) {
        banner("STEP 1", "                                     loading reads from file");
        const std::string path = savedReadsPath(o);
        if (const int rc = sage2gpu_load_saved_reads(ctx, path.c_str(), o.minOverlap)) {
            if (rc == SAGE2GPU_ERR_FORMAT) savedReadsError(path, sage2gpu_last_error(ctx));
            printError(rc == SAGE2GPU_ERR_IO ? "OPEN_FILE" : "CUDA", sage2gpu_last_error(ctx));
        }
        logStream << "Function loadReadsFromFile() in " << seconds_since(t0) << " sec.\n";
    } else {
        banner("STEP 1", "                                          organizing reads");
        Uploader up({ ctx }, o.minOverlap);
        if (!o.listInput.empty()) loadFromList(up, o.listInput);
        else readDataset(up, o.fileInput, "");
        logStream << "Parsed and uploaded in " << seconds_since(t0) << " sec.\n";
        auto t1 = std::chrono::steady_clock::now();
        up.finish();
        logStream << "Function organizeReads() in " << seconds_since(t1) << " sec.\n";
    }
    sage2gpu_get_counters(ctx, &cnt);
    logStream << std::setw(20) << "Total reads: " << cnt.total_reads << "\n";
    logStream << std::setw(20) << "Good reads: " << cnt.good_reads << "\n";
    logStream << std::setw(20) << "Bad reads: " << cnt.total_reads - cnt.good_reads << "\n";
    logStream << "\t" << std::setw(21) << "Average read length: " << cnt.avg_len << "\n";
    logStream << "\tNumber of unique reads: " << cnt.unique_reads << "\n";
    logStream.flush();
    const bool saveReads = (o.maxStep <= 3 || o.saveAll || o.maxStep > 3) &&      // steps 4-7 continue from the files
                           (!restart || writeReadsAfterRestart(o, base));
    if (saveReads) {
        auto t = std::chrono::steady_clock::now();
        if (sage2gpu_write_reads(ctx, (base + ".reads").c_str()) != 0) printError("OPEN_FILE", sage2gpu_last_error(ctx));
        logStream << "Function saveReadsInFile in " << seconds_since(t) << " sec.\n";
    }
    if (o.maxStep == 1) { sage2gpu_destroy(ctx); return 0; }

    // ---- step 2 -------------------------------------------------------------------------------------
    banner("STEP 2", "                                         building hash table");
    t0 = std::chrono::steady_clock::now();
    if (sage2gpu_build_hash_table(ctx) != 0) printError("CUDA", sage2gpu_last_error(ctx));
    sage2gpu_get_counters(ctx, &cnt);
    logStream << "\tHash string length: " << cnt.hash_len << "\n";
    logStream << "\tSize of hash table: " << cnt.table_capacity << " slots, " << cnt.distinct_keys << " distinct keys\n";
    logStream << "\tNumber of hashes over threshold: " << cnt.keys_over_threshold << "\n";
    logStream << "Function hashPrefixesAndSuffix() in " << seconds_since(t0) << " sec.\n";
    if (o.maxStep == 2 || o.saveAll)
        logStream << "NOTE: " << o.prefixName << ".hashTable is not written (see sage2gpu_main.cpp header).\n";
    logStream.flush();
    if (o.maxStep == 2) { sage2gpu_destroy(ctx); return 0; }

    // ---- step 3 -------------------------------------------------------------------------------------
    banner("STEP 3", "                                      building overlap graph");
    t0 = std::chrono::steady_clock::now();
    if (sage2gpu_build_overlap_graph(ctx) != 0) printError("CUDA", sage2gpu_last_error(ctx));
    sage2gpu_get_counters(ctx, &cnt);
    logStream << "\tTotal reads contained by extension: " << cnt.contained_ext << "\n";
    logStream << "\tTotal reads contained by size: " << cnt.contained_size << "\n";
    logStream << "\tTotal reads left to explore: " << cnt.left_to_explore << "\n";
    logStream << "\tTotal edges inserted: " << cnt.edges_inserted_c << "\n";
    logStream << "\tTotal transitive edges removed: " << cnt.transitive_removed << "\n";
    logStream << "\tEdges in the overlap graph: " << cnt.n_edges << "\n";
    logStream << "Functions buildInitialOverlapGraph() + buildOverlapGraphEconomy() + sortEconomyGraph() in " << seconds_since(t0) << " sec.\n";
    sage2gpu_timers tm;
    sage2gpu_get_timers(ctx, &tm);
    logStream << "\tDevice ms: ingest " << tm.ingest << ", sort " << tm.sort_reads << ", table " << tm.build_table << ", phase A "
              << tm.phase_a << ", phase B " << tm.phase_b << ", phase C " << tm.phase_c_dev << " + host " << tm.phase_c_host
              << ", edges " << tm.sort_edges << "\n";
    {
        auto t = std::chrono::steady_clock::now();
        if (sage2gpu_write_graph3(ctx, (base + ".graph3").c_str()) != 0) printError("OPEN_FILE", sage2gpu_last_error(ctx));
        logStream << "Function saveOverlapGraphInFile in " << seconds_since(t) << " sec.\n";
    }
    if (o.gfa) saveGfa(ctx, base);
    logStream.flush();
    sage2gpu_destroy(ctx);
    if (o.maxStep <= 3) return 0;

    // ---- steps 4-7: the reference's own, from the files above --------------------------------------------
    if (o.referenceBin.empty()) {
        logStream << "Steps 4-" << o.maxStep << " are the reference's: run `SAGE2 -m 4 -i " << o.prefixName << " ...` (or give --reference).\n";
        std::cout << "sage2gpu: steps 1-3 done (" << base << ".reads, " << base << ".graph3); continue with SAGE2 -m 4 -i " << o.prefixName << "\n";
        return 0;
    }
    logStream << "Running " << o.referenceBin << " -m 4 for steps 4-" << o.maxStep << ".\n";
    logStream.close();
    return runReference(o, 4);
}
