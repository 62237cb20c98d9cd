// core.cuh -- host/device primitives of libsage2gpu (record layout, keys, compares, table slots,
// the unique-extension state machine).  Everything here is pure bit arithmetic on 64-bit words so
// that the same code is exercised on the CPU by tests/ (compiled with g++) and on sm_100a by the
// kernels.  Reference citations are relative to /root/reference.
//
// READ RECORD (device layout).  Every read is a fixed-stride record of SW 64-bit words,
// WORD-BIG-ENDIAN: base p lives in word p/32 at bit 62-2*(p%32) (A0 C1 G2 T3, the codes of
// utils.cpp:96-119), unused sequence bits are 0, and the low 16 bits of the LAST word hold the read
// length.  SW = ceil((2*maxLen+16)/64), so sequence bits and the length never overlap.  Comparing two
// records word by word as unsigned integers is exactly Read::operator< (readLoader.cpp:11-18 /
// utils.cpp:224-242: zero-padded bytes first, then length), so the record is its own sort key.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define SG_HD __host__ __device__ __forceinline__
#else
#define SG_HD inline
#endif

namespace sg {

typedef uint64_t u64;
typedef uint32_t u32;

constexpr int kMaxWords = 32;          // <= 1016 bases per read
constexpr int kHashThreshold = 100;    // hashTable.cpp:76
constexpr u32 kConnectionsLimit = 300; // economyGraph.cpp:43

SG_HD int words_for_len(int max_len) { return (2 * max_len + 16 + 63) / 64; }
// F / RC storage stride in words: whole 32-byte sectors, a power-of-two number of them per record, so
// that a record never straddles a 128-byte line and 1/2/4/8 lanes fetch it with one 256-bit load each.
SG_HD int storage_words(int SW) { return SW <= 4 ? 4 : (SW <= 8 ? 8 : (SW <= 16 ? 16 : 32)); }
SG_HD int rec_len(const u64 *rec, int SW) { return (int)(rec[SW - 1] & 0xFFFFull); }
SG_HD int hash_len_for(int min_overlap) { return min_overlap > 64 ? 64 : min_overlap; }  // hashTable.cpp:78-81

// 32 bases starting at base s, left aligned (bases past the record end read as 0 / garbage that
// callers shift or mask away).
SG_HD u64 window32(const u64 *X, int SW, int s)
{
    const int i = s >> 5, sh = (s & 31) * 2;
    const u64 a = i < SW ? X[i] : 0ull;
    if (sh == 0) return a;
    const u64 b = (i + 1) < SW ? X[i + 1] : 0ull;
    return (a << sh) | (b >> (64 - sh));
}

// bases [s, s+n), 1 <= n <= 32, as a right-aligned big-endian 2-bit integer == get64BitInt
// (utils.cpp:189-207).
SG_HD u64 get_bases(const u64 *X, int SW, int s, int n) { return window32(X, SW, s) >> (64 - 2 * n); }

// get64Bit2Int (utils.cpp:171-187): v1 = last min(h,32) bases, v0 = leading h-32 bases.
SG_HD void extract_key(const u64 *X, int SW, int j, int h, u64 &v0, u64 &v1)
{
    if (h <= 32) { v0 = 0; v1 = get_bases(X, SW, j, h); }
    else { v0 = get_bases(X, SW, j, h - 32); v1 = get_bases(X, SW, j + h - 32, 32); }
}

// X[start+t] == Y[t] for t in [0, ov), ov = min(lenY, lenX-start).  `contained` = Y ends at or
// before X's end.  With the first h bases known equal (key match) this is compareStringInBytes /
// compareStringInBytesPrevious (economyGraph.cpp:712-808); comparing from t=0 also re-verifies the key.
SG_HD bool overlap_equal(const u64 *X, int lenX, int start, const u64 *Y, int lenY, int SW, bool &contained)
{
    const int rem = lenX - start;
    contained = lenY <= rem;
    const int ov = contained ? lenY : rem;
    for (int w = 0; w * 32 < ov; ++w) {
        const u64 xs = window32(X, SW, start + 32 * w);
        const int nb = ov - 32 * w;
        const u64 m = nb >= 32 ? ~0ull : ~(~0ull >> (2 * nb));
        if ((xs ^ Y[w]) & m) return false;
    }
    return true;
}

// reverse the order of the 32 two-bit groups of a word
SG_HD u64 rev2(u64 w)
{
#if defined(__CUDA_ARCH__)
    w = __brevll(w);
    return ((w >> 1) & 0x5555555555555555ull) | ((w & 0x5555555555555555ull) << 1);
#else
    w = ((w >> 2) & 0x3333333333333333ull) | ((w & 0x3333333333333333ull) << 2);
    w = ((w >> 4) & 0x0F0F0F0F0F0F0F0Full) | ((w & 0x0F0F0F0F0F0F0F0Full) << 4);
    return __builtin_bswap64(w);
#endif
}

// Record of the reverse complement (utils.cpp:73-91 on packed words): reverse all 2-bit groups of
// the SW*64-bit string, complement, shift the sequence back to the top, re-attach the length.
// Word w of it depends on two words of F only, so lanes that share a record can each produce their own words.
SG_HD u64 revcomp_word(const u64 *F, int SW, int len, int w)
{
    const int sh = 64 * SW - 2 * len;     // >= 16
    const int q = sh >> 6, r = sh & 63;
    const int i0 = w + q, i1 = w + q + 1;
    const u64 a = i0 < SW ? rev2(~F[SW - 1 - i0]) : 0ull;
    const u64 b = i1 < SW ? rev2(~F[SW - 1 - i1]) : 0ull;
    const u64 x = r == 0 ? a : ((a << r) | (b >> (64 - r)));
    return w == SW - 1 ? x | (u64)len : x;
}
SG_HD void revcomp_record(const u64 *F, u64 *R, int SW, int len)
{
    for (int w = 0; w < SW; ++w) R[w] = revcomp_word(F, SW, len, w);
}

// ---- prefix/suffix table ----------------------------------------------------------------------
// An entry is (readId0 << 2) | type with readId0 = readId-1 and type as in hashTable.cpp:98-105:
// 0 fwd prefix, 1 fwd suffix, 2 revcomp prefix, 3 revcomp suffix.  Entries are sorted by
// (key, readId, type) so that every key's entries are contiguous and already in the reference's
// bucket order (insertion order, hashTable.cpp:94-109).  The open-addressing index maps
// key -> bucket with one 64-bit slot per distinct key:
//   [63:40] tag: the low SG_SLOT_TAG_BITS (24) bits of the key hash   [39:33] min(count,127)
//   [32:0]  count == 1: the entry itself (no second hop);  count > 1: offset of the first entry
// A slot is never 0 when occupied (count >= 1).  count >= 100 means "masked" (hashTable.cpp:116-121).
// Slots are grouped in 32-byte SECTORS of 4: a key's home is a sector (one DRAM sector per probe),
// insertion and search walk the 4 slots of a sector in order, then the next sector.
SG_HD u64 mix64(u64 x)
{
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
    return x;
}
SG_HD u64 hash_key(u64 v0, u64 v1) { return mix64(v1 ^ mix64(v0 + 0x9e3779b97f4a7c15ull)); }
SG_HD u64 mulhi64(u64 a, u64 b)
{
#if defined(__CUDA_ARCH__)
    return __umul64hi(a, b);
#else
    return (u64)(((unsigned __int128)a * b) >> 64);
#endif
}
constexpr int kSlotsPerSector = 4;
SG_HD u64 home_sector(u64 hsh, u64 nsec) { return mulhi64(hsh, nsec); }
// Bits of the key hash a slot keeps as its tag.  The product uses all 24; the test suite builds variants with fewer
// (-DSG_SLOT_TAG_BITS=0 / 8) so that tag collisions, which every search must resolve, happen on small data sets too.
#ifndef SG_SLOT_TAG_BITS
#define SG_SLOT_TAG_BITS 24
#endif
static_assert(SG_SLOT_TAG_BITS >= 0 && SG_SLOT_TAG_BITS <= 24, "a slot has room for a tag of at most 24 bits");
SG_HD u64 slot_tag(u64 hsh) { return hsh & ((1ull << SG_SLOT_TAG_BITS) - 1); }
SG_HD u64 slot_encode(u64 hsh, u64 count, u64 payload)
{
    return (slot_tag(hsh) << 40) | ((count > 127 ? 127ull : count) << 33) | payload;
}
SG_HD u64 slot_get_tag(u64 s) { return s >> 40; }
SG_HD u32 slot_get_count(u64 s) { return (u32)((s >> 33) & 127); }
SG_HD u64 slot_get_payload(u64 s) { return s & 0x1FFFFFFFFull; }

// Key of table entry `type` of a read (hashTable.cpp:98-101)
SG_HD void entry_key(const u64 *F, const u64 *RC, int SW, int len, int h, int type, u64 &v0, u64 &v1)
{
    const u64 *X = (type & 2) ? RC : F;
    extract_key(X, SW, (type & 1) ? len - h : 0, h, v0, v1);
}

// ---- phase A: the unique-extension state machine (economyGraph.cpp:86-439) -----------------------
struct ExtState {
    u32 Rid, Rtype, Rlen;                 // rightExtension[i]
    u32 Lid, Ltype, Llen;                 // leftExtension[i]
    int prevJR, prevLenR, prevTypeR;      // prevLengthRight (= window j), previous read's length
    int prevPL, prevLenL, prevTypeL;      // prevLengthLeft  (= len1-j-h)
    int markAmbigR, markFirstR, markAmbigL, itsAmbigR, itsAmbigL;
    u32 connections;
};
SG_HD void ext_init(ExtState &s)
{
    s.Rid = s.Rtype = s.Rlen = 0; s.Lid = s.Ltype = s.Llen = 0;
    s.prevJR = s.prevLenR = s.prevTypeR = 0; s.prevPL = s.prevLenL = s.prevTypeL = 0;
    s.markAmbigR = s.markFirstR = s.markAmbigL = s.itsAmbigR = s.itsAmbigL = 0;
    s.connections = 0;
}
SG_HD void ext_new_window(ExtState &s) { s.markAmbigR = 0; s.markAmbigL = 0; s.markFirstR = 0; }   // :86-88

SG_HD void copy_rec(u64 *dst, const u64 *src, int SW) { for (int w = 0; w < SW; ++w) dst[w] = src[w]; }

// Accepted right hit (hash types 0 / 2): Q = partner oriented like read i (fwd for type 0, revcomp
// for type 2), t01 = 0 / 1.  prevRec holds the oriented record of the current "previous" read.
// economyGraph.cpp:94-276.
SG_HD void ext_right_hit(ExtState &s, u64 *prevRec, const u64 *Q, int SW, u32 read2, int t01, int j, int len1, int len2)
{
    s.connections++;
    if (s.Rid == 0) {
        s.Rid = read2; s.Rtype = (u32)t01; s.Rlen = (u32)(len2 - (len1 - j));
        s.prevTypeR = t01; s.prevJR = j; s.prevLenR = len2; copy_rec(prevRec, Q, SW);
        s.markAmbigR = 1; s.markFirstR = 1;
        return;
    }
    bool c;
    if (overlap_equal(prevRec, s.prevLenR, j - s.prevJR, Q, len2, SW, c)) {
        if (s.markAmbigR == 1) {
            if (len2 > s.prevLenR) {
                if (s.markFirstR == 1) { s.Rid = read2; s.Rtype = (u32)t01; s.Rlen = (u32)(len2 - (len1 - j)); }
                s.prevTypeR = t01; s.prevJR = j; s.prevLenR = len2; copy_rec(prevRec, Q, SW);
            }
        } else {
            s.prevTypeR = t01; s.prevJR = j; s.prevLenR = len2; copy_rec(prevRec, Q, SW);
            s.markAmbigR = 1;
        }
    } else s.itsAmbigR = 1;
}

// Accepted left hit (hash types 1 / 3): Q = partner oriented like revcomp(read i) (revcomp for type 1,
// fwd for type 3), t01 = 0 / 1, p = len1-j-h.  economyGraph.cpp:279-437.
SG_HD void ext_left_hit(ExtState &s, u64 *prevRec, const u64 *Q, int SW, u32 read2, int t01, int j, int h, int len1, int len2)
{
    const int p = len1 - j - h;
    s.connections++;
    if (s.Lid == 0) {
        s.Lid = read2; s.Ltype = (u32)t01; s.Llen = (u32)(len2 - j - h);
        s.prevTypeL = t01; s.prevPL = p; s.prevLenL = len2; copy_rec(prevRec, Q, SW);
        s.markAmbigL = 1;
        return;
    }
    bool c;
    if (overlap_equal(Q, len2, s.prevPL - p, prevRec, s.prevLenL, SW, c)) {
        if (s.markAmbigL == 1) {
            if (len2 > s.prevLenL) {
                s.Lid = read2; s.Ltype = (u32)t01; s.Llen = (u32)(len2 - j - h);
                s.prevTypeL = t01; s.prevPL = p; s.prevLenL = len2; copy_rec(prevRec, Q, SW);
            }
        } else {
            s.Lid = read2; s.Ltype = (u32)t01; s.Llen = (u32)(len2 - j - h);
            s.prevTypeL = t01; s.prevPL = p; s.prevLenL = len2; copy_rec(prevRec, Q, SW);
            s.markAmbigL = 1;
        }
    } else s.itsAmbigL = 1;
}

// Extension record handed to phase B: [31:0] read id (1-based, 0 = none), bit 32 strand type,
// [54:33] 22-bit overhang (ExtensionTable, economyGraph.h:24-30).
SG_HD u64 ext_pack(u32 id, u32 type, u32 len) { return (u64)id | ((u64)(type & 1) << 32) | ((u64)(len & 0x3FFFFFu) << 33); }
SG_HD u32 ext_id(u64 e) { return (u32)e; }
SG_HD u32 ext_type(u64 e) { return (u32)(e >> 32) & 1u; }
SG_HD u32 ext_length(u64 e) { return (u32)(e >> 33) & 0x3FFFFFu; }

// ---- edges --------------------------------------------------------------------------------------
// Canonical edge record (from < to): w0 = from<<32 | to (1-based ids), w1 = type<<20 | overhang
// (20-bit EconomyEdge::length, economyGraph.h:14-22).  Sorting by (w0,w1) is compareIdBased
// (economyGraph.cpp:875-893) applied to list[from]; only entries with to > from are consumed by
// convertGraph (overlapGraph.cpp:103).
SG_HD u32 reverse_edge_type(u32 t) { return t == 0 ? 3u : (t == 3 ? 0u : t); }     // utils.cpp:212-219
struct EdgeRec { u64 w0, w1; };
// insertEdgeEconomy(u, v, delta, type) (economyGraph.cpp:813-849) seen from the smaller endpoint.
SG_HD EdgeRec edge_canonical(u32 u, u32 v, u32 delta, u32 type, u32 len_u, u32 len_v)
{
    EdgeRec e;
    if (u < v) {
        e.w0 = ((u64)u << 32) | v; e.w1 = ((u64)type << 20) | (delta & 0xFFFFFu);
    } else {
        const u32 delta2 = len_u - (len_v - delta);
        e.w0 = ((u64)v << 32) | u; e.w1 = ((u64)reverse_edge_type(type) << 20) | (delta2 & 0xFFFFFu);
    }
    return e;
}

// ---- gating and candidate encoding shared by phase A / phase C --------------------------------------
SG_HD bool gate_right(int j, int len1, int k) { return j <= (int)(uint16_t)(len1 - k); }   // economyGraph.cpp:94,187
SG_HD bool gate_left(int j, int k, int h) { return j >= (int)(uint16_t)(k - h); }          // :279,359
// entry type -> which strand record of the partner is compared (types 1,2 use the reverse complement)
SG_HD bool partner_uses_rc(int type) { return type == 1 || type == 2; }
// phase-C candidate: read2(1-based)<<32 | edgeType<<20 | overhang20.  Hash type 0->edge 3, 1->0, 2->2,
// 3->1 and the overhang formulas of economyGraph.cpp:607-626.
SG_HD u64 candidate_record(int type, int j, int h, int len1, int len2, u32 rid2_0based)
{
    const u32 etype = type == 0 ? 3u : type == 1 ? 0u : type == 2 ? 2u : 1u;
    const int ovlp = (type & 1) ? len2 - j - h : len2 - (len1 - j);
    return ((u64)(rid2_0based + 1) << 32) | ((u64)etype << 20) | ((u32)ovlp & 0xFFFFFu);
}

// ---- multi-GPU: reads (as query sources) are block-partitioned by id, the last rank's slice may be short ----
SG_HD u64 partition_chunk(u64 U, int world) { return world <= 1 ? U : (U + (u64)world - 1) / (u64)world; }

// ---- multi-GPU, sharded table (SURVEY 8(e)): shard g owns the keys with key_owner(hash) == g.  The owner comes
// from hash bits 24..33: disjoint from the slot tag (bits 0..23) and from the bits home_sector() consumes.
constexpr int kMaxWorld = 64;
SG_HD int key_owner(u64 hsh, int world) { return world <= 1 ? 0 : (int)(((hsh >> 24) & 0x3FFull) % (u64)world); }
// A complete table assembled from `shards` key-hash shards laid out back to back (nsec sectors each): a probe starts in
// the shard that owns its key and wraps inside it.  shards == 1: the plain table.
SG_HD u64 shard_base_sector(u64 hsh, u64 nsec, int shards) { return shards <= 1 ? 0ull : (u64)key_owner(hsh, shards) * nsec; }
// Answer of an owner to one routed window probe = a slot word without its tag: count << 33 | payload, payload =
// the only entry (count 1), a representative entry (count >= 100, tag probes only) or the offset of the bucket's
// run in the entry stream the owner returns alongside.  0 = absent.
SG_HD u64 answer_encode(u32 count, u64 payload) { return ((u64)(count > 127 ? 127u : count) << 33) | payload; }

// ---- phase B (economyGraph.cpp:455-480) ---------------------------------------------------------------
// State after phase A.  The reference writes 6 from any thread (:735) and 5 from the owner (:444); a
// 1-thread run resolves that race by time order, reproduced here: the containing scan with the largest
// id wrote last unless the read's own iteration (which writes 5 at its end) came later.
SG_HD uint8_t state_after_a(u32 id /*1-based*/, u32 cont_max, uint8_t f5)
{
    if (cont_max) return (f5 && id >= cont_max) ? 5 : 6;
    return f5 ? 5 : 0;
}
// reciprocal unique extension on both sides (:460); i is 0-based
SG_HD bool phase_b_qualifies(const u64 *extR, const u64 *extL, u64 i)
{
    const u32 id = (u32)i + 1;
    const u64 L = extL[i], R = extR[i];
    if (ext_length(L) == 0 || ext_length(R) == 0) return false;
    const u32 l = ext_id(L) - 1, r = ext_id(R) - 1;
    const bool lrec = ext_id(extR[l]) == id || ext_id(extL[l]) == id;
    const bool rrec = ext_id(extR[r]) == id || ext_id(extL[r]) == id;
    return lrec && rrec;
}
// Edges read i (state 4) inserts: i->L and i->R unless the target was already state 4 when i was
// visited, i.e. unless the target qualifies too and has a smaller id (:462-473).  Returns 0..2 records.
SG_HD int phase_b_edges(const u64 *extR, const u64 *extL, const uint8_t *explored, const uint16_t *len, u64 i, EdgeRec e[2])
{
    int n = 0;
    if (explored[i] != 4) return 0;
    const u32 id = (u32)i + 1;
    const u64 L = extL[i], R = extR[i];
    const u32 lid = ext_id(L), rid = ext_id(R);
    if (!(explored[lid - 1] == 4 && lid < id))
        e[n++] = edge_canonical(id, lid, ext_length(L), ext_type(L) == 0 ? 0u : 1u, len[i], len[lid - 1]);
    if (!(explored[rid - 1] == 4 && rid < id))
        e[n++] = edge_canonical(id, rid, ext_length(R), ext_type(R) == 0 ? 3u : 2u, len[i], len[rid - 1]);
    return n;
}

}  // namespace sg
