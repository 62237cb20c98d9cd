// device_utils.cuh -- error handling, stream-ordered allocation, exclusive scan and LSD radix sort.
// Hand-written for sm_100a (no CUB/Thrust on the product path).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <algorithm>
#include <stdexcept>
#include <string>
#include <vector>

namespace sg {

typedef uint64_t u64;
typedef uint32_t u32;

struct CudaError : public std::runtime_error {
    explicit CudaError(const std::string &m) : std::runtime_error(m) {}
};

#define SG_CUDA(call)                                                                           \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess)                                                                 \
            throw sg::CudaError(std::string(#call) + " failed: " + cudaGetErrorString(e__) +    \
                                " at " + __FILE__ + ":" + std::to_string(__LINE__));            \
    } while (0)

#define SG_CHECK(cond, msg)                                                                     \
    do {                                                                                        \
        if (!(cond)) throw sg::CudaError(std::string(msg) + " (" #cond ") at " + __FILE__ + ":" + \
                                         std::to_string(__LINE__));                             \
    } while (0)

// Workspace arena: the temporaries of one stage are bump-allocated from a few large grow-only blocks and the
// arena is rewound when the stage ends.  (Cycling hundreds of MB .. GB of temporaries through the stream-ordered
// pool every call made cudaMallocAsync map fresh memory at unpredictable times: stalls of 0.1 - 5 s at 33 M reads.)
struct Arena {
    struct Block { char *p; size_t cap; };
    std::vector<Block> blocks;
    size_t used = 0;            // bytes taken from the last block
    size_t peak = 0;            // high-water mark of the current scope over all blocks
    bool tight = false;         // low-memory mode: blocks of exactly the size asked for, everything released at the end of the stage
    static size_t round(size_t b) { return (b + 255) & ~(size_t)255; }
    size_t total() const { size_t t = 0; for (const Block &b : blocks) t += b.cap; return t; }
    void *take(size_t bytes)
    {
        bytes = round(bytes ? bytes : 1);
        if (blocks.empty() || used + bytes > blocks.back().cap) {
            size_t cap = tight ? std::max<size_t>(bytes, (size_t)64 << 20) : std::max<size_t>(bytes, std::max<size_t>((size_t)64 << 20, total() / 2));
            char *p = nullptr;
            SG_CUDA(cudaMalloc((void **)&p, cap));
            blocks.push_back(Block{ p, cap });
            used = 0;
        }
        void *r = blocks.back().p + used;
        used += bytes;
        return r;
    }
    void give_back(void *p, size_t bytes)      // only the most recent allocation is really returned
    {
        bytes = round(bytes ? bytes : 1);
        if (!blocks.empty() && (char *)p + bytes == blocks.back().p + used) used -= bytes;
    }
    // end of a stage: rewind; several blocks (growth during this stage) are merged into one
    void reset(cudaStream_t st)
    {
        if (tight) {        // large workspaces go back to the driver, small ones (the routed batches of the sharded table) stay
            if (total() > ((size_t)1 << 30)) { cudaStreamSynchronize(st); destroy(); }
            used = 0;
            if (blocks.size() <= 1) return;
        }
        if (blocks.size() > 1) {
            const size_t want = total() + total() / 4;
            cudaStreamSynchronize(st);
            for (Block &b : blocks) cudaFree(b.p);
            blocks.clear();
            char *p = nullptr;
            if (cudaMalloc((void **)&p, want) == cudaSuccess) blocks.push_back(Block{ p, want });
            else cudaGetLastError();
        }
        used = 0;
    }
    void destroy()
    {
        for (Block &b : blocks) cudaFree(b.p);
        blocks.clear();
        used = 0;
    }
};

inline Arena *&current_arena() { static thread_local Arena *a = nullptr; return a; }

struct ArenaScope {
    Arena *prev;
    Arena &a;
    cudaStream_t st;
    ArenaScope(Arena &arena, cudaStream_t s) : prev(current_arena()), a(arena), st(s) { current_arena() = &a; }
    ~ArenaScope() { current_arena() = prev; if (!prev) a.reset(st); }
};

// Device buffer.  Long-lived buffers of a context (`persistent`) come from the stream-ordered pool and are
// grow-only; everything else comes from the arena of the running stage.
template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0, cap = 0;      // n = elements in use, cap = elements allocated
    cudaStream_t s = nullptr;
    bool persistent = false, from_arena = false;
    DevBuf() {}
    DevBuf(size_t count, cudaStream_t st) { alloc(count, st); }
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : p(o.p), n(o.n), cap(o.cap), s(o.s), persistent(o.persistent), from_arena(o.from_arena) { o.p = nullptr; o.n = 0; o.cap = 0; }
    DevBuf &operator=(DevBuf &&o) noexcept
    {
        if (this != &o) {
            release();
            p = o.p; n = o.n; cap = o.cap; s = o.s; from_arena = o.from_arena;      // `persistent` is a property of the holder
            o.p = nullptr; o.n = 0; o.cap = 0;
        }
        return *this;
    }
    ~DevBuf() { release(); }
    // Contents are undefined.  A persistent buffer that is already large enough is kept.
    void alloc(size_t count, cudaStream_t st)
    {
        if (p && !from_arena && cap >= count && s == st) { n = count; return; }
        release();
        s = st; n = count; cap = count ? count : 1;
        Arena *a = persistent ? nullptr : current_arena();
        if (a) { p = (T *)a->take(cap * sizeof(T)); from_arena = true; }
        else { SG_CUDA(cudaMallocAsync((void **)&p, cap * sizeof(T), st)); from_arena = false; }
    }
    void release()
    {
        if (!p) return;
        if (from_arena) { if (Arena *a = current_arena()) a->give_back(p, cap * sizeof(T)); }
        else cudaFreeAsync(p, s);
        p = nullptr; n = 0; cap = 0; from_arena = false;
    }
    size_t bytes() const { return n * sizeof(T); }
};

// page-locked host staging buffer of a context (grow-only): device -> host copies into it run at PCIe speed and do not
// pass through the driver's bounce buffers
struct PinnedBuf {
    void *p = nullptr;
    size_t cap = 0;
    void *ensure(size_t bytes)
    {
        if (bytes > cap) {
            if (p) cudaFreeHost(p);
            p = nullptr; cap = 0;
            const size_t want = bytes + bytes / 4 + 4096;
            SG_CUDA(cudaHostAlloc(&p, want, cudaHostAllocDefault));
            cap = want;
        }
        return p;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// give the freed blocks of the stream-ordered pool back to the driver (low-memory mode: the workspace arena and other
// allocators can then use them)
inline void trim_default_pool(int device, cudaStream_t st)
{
    cudaStreamSynchronize(st);
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
}

constexpr int kSMs = 148;   // B200

// every kernel launch of the library is followed by SG_LAUNCHED(): error check + launch count
// (bench.py reports the count as `gpu_launches`).
inline unsigned long long &launch_counter() { static unsigned long long n = 0; return n; }
#define SG_LAUNCHED()                     \
    do {                                  \
        ++sg::launch_counter();           \
        SG_CUDA(cudaGetLastError());      \
    } while (0)

// SAGE2GPU_STAGE_STATS set: stages print the sizes their cost depends on to stderr (tools/stage_kernels.py collects them)
inline bool stage_stats_enabled() { return getenv("SAGE2GPU_STAGE_STATS") != nullptr; }

inline unsigned grid_for(u64 n, unsigned block, unsigned per_thread = 1)
{
    u64 g = (n + (u64)block * per_thread - 1) / ((u64)block * per_thread);
    if (g == 0) g = 1;
    SG_CHECK(g < 0x7FFFFFFFull, "grid too large");
    return (unsigned)g;
}

// exclusive prefix sum of n u32 values (in may alias out); returns the grand total through
// d_total (device pointer, may be null).  Sums must fit in 32 bits.
void exclusive_scan_u32(const u32 *in, u32 *out, u64 n, u32 *d_total, cudaStream_t st);

// OR / AND of n 64-bit keys -> d_or_and[0], d_or_and[1] (device); used to skip constant digits.
void reduce_or_and_u64(const u64 *keys, u64 n, u64 *d_or_and, cudaStream_t st);

// Stable LSD radix sort of n records by bits [lo,hi) of keyA (use_b=false) or keyB (use_b=true).
// A record is (keyA[, keyB][, val]); null pointers mean "that column does not exist".  Buffers
// ping-pong between (a0,b0,v0) and (a1,b1,v1); returns 0 if the result is in set 0, else 1.
struct SortCols {
    u64 *a[2];
    u64 *b[2];
    u32 *v[2];
};
int radix_sort_bits(SortCols &c, int cur, u64 n, bool use_b, int lo, int hi, cudaStream_t st);

// Convenience: sort by all VARYING bits of the chosen key column (one host sync to read OR/AND).
int radix_sort_varying(SortCols &c, int cur, u64 n, bool use_b, cudaStream_t st);

// GB/s of uniformly random `granule_bytes` gathers over `footprint_bytes` of HBM (best of 3 after warm-up).
float gather_bench(u64 footprint_bytes, int granule_bytes, u64 n_loads, int mode, cudaStream_t st);

}  // namespace sg
