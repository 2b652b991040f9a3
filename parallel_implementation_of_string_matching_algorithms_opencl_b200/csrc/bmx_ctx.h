// bmx_ctx.h -- per (host thread, device) context behind the convenience entry points: one cached scanner, two
// streams, events, pinned bounce buffers and two cached device buffers (text, positions).  Not installed.
//
// Device memory policy: the library never touches the attributes of the device's default memory pool and never
// sizes a buffer by the worst case (8 bytes per text byte).  The cached buffers are plain cudaMalloc blocks that
// grow on demand, are reused by later calls of the same thread and are given back by bmx_release_memory() or
// when the thread exits.
#pragma once

#include <cuda_runtime.h>

#include <algorithm>
#include <vector>

#include "bmx_internal.h"
#include "bmx_scanner.h"

#define BMX_CUDA(call)                                                                                   \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            (void)cudaGetLastError();                                                                    \
            return bmx::fail(e_ == cudaErrorMemoryAllocation ? BMX_E_NOMEM : BMX_E_CUDA, "%s: %s", #call, \
                             cudaGetErrorString(e_));                                                    \
        }                                                                                                \
    } while (0)

namespace bmx {

constexpr int kMaxDevices = 64;
constexpr int kBounce = 3;
constexpr int64_t kSmallSpec = 8192;   // positions read back together with the count (64 KiB)

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct ThreadCtx {
    int device = -1;
    bmx_scanner *scanner = nullptr;
    cudaStream_t copy_stream = nullptr, scan_stream = nullptr;
    std::vector<cudaEvent_t> events;
    unsigned char *bounce[kBounce] = {nullptr, nullptr, nullptr};
    size_t bounce_bytes = 0;
    DevBuf text, pos, misc, aux;
    int64_t *h_small = nullptr;   // pinned landing area for the speculative result read of small host texts (kSmallSpec entries)
    ThreadCtx() = default;
    ThreadCtx(const ThreadCtx &) = delete;
    ThreadCtx &operator=(const ThreadCtx &) = delete;
    ~ThreadCtx();            // a host thread that exits gives everything back
    void release_buffers();  // text / positions / bounce buffers only (bmx_release_memory)
};

// ---- argument checks shared by the entry points (bmx_abi.cu).  Each returns BMX_OK or the code of bmx::fail.
int check_device(int device);
int check_text(const void *text, int64_t n, const char *who);   // n >= 0, and a text pointer unless n == 0
int check_pattern(int32_t m);                                    // 1 <= m <= BMX_MAX_PATTERN
// npat >= 0 with pats / ms / counts; then every pattern non-NULL, 1 <= ms[k] <= BMX_MAX_PATTERN, a cap for every
// output buffer; counts[k] is zeroed as the loop passes it.
int check_pattern_set(int32_t npat, const char *const *pats, const int32_t *ms, int64_t *const *outs, const int64_t *caps,
                      uint64_t *counts, const char *who);

int get_ctx(int device, ThreadCtx **out);   // the calling thread's context for `device`
int current_ctx(ThreadCtx **out);           // ... for the calling thread's current device
int ensure_streams(ThreadCtx &c, size_t nevents);
// Grows b to at least `bytes` (never shrinks).  The old block may still be in use by work enqueued on the
// context's streams, so they are drained before it is freed.  NOMEM leaves b empty.
int ensure_buf(ThreadCtx &c, DevBuf &b, size_t bytes);
int scanner_begin_find(bmx_scanner *s, void *stream);   // find-first search: count-only kernels + early stop (bmx_abi.cu)
// One whole search with the scanner: set_pattern, begin, one scan of d_text[0..n), finish (bmx_abi.cu).
int search_once(bmx_scanner *s, const char *pat, int32_t m, int32_t variant, const void *d_text, int64_t n, int64_t pos_base,
                int64_t *d_pos, int64_t pos_cap, uint64_t *count, bmx_stats *stats, void *stream);

// The position buffer of a search follows its count (DESIGN §2): a first guess of one hit per 64 bytes, at least
// 1 Mi entries, never more than the want_cap positions the caller can use ...
inline int64_t first_pos_cap(int64_t n, int32_t m, int64_t want_cap)
{
    return std::max<int64_t>(0, std::min<int64_t>({want_cap, n - m + 1, std::max<int64_t>(int64_t(1) << 20, n / 64)}));
}
// ... or the room c.pos already holds, if that is more.
inline int64_t first_pos_room(const ThreadCtx &c, int64_t n, int32_t m, int64_t want_cap)
{
    const int64_t cap = first_pos_cap(n, m, want_cap), owned = (int64_t)(c.pos.cap / 8);
    return owned > cap ? std::min(want_cap, owned) : cap;
}

// One shard of a host text through the calling GPU's context (bmx_host.cu, used by bmx_multi.cu).
int ingest_shard(ThreadCtx &ctx, int device, const char *text, int64_t n, const char *pat, int32_t m, int64_t pos_base,
                 int64_t want_cap, uint64_t *count, int64_t *dev_cap);
// A host text copied once into ctx.text (the chunked ingest without a scan); NOMEM when it does not fit (bmx_host.cu).
int copy_text_resident(ThreadCtx &ctx, const char *text, int64_t n);

// Per-range counts, offsets and positions of host ranges over a host text (bmx_ranges.cu).  The ranges are checked
// (inside [0, n], begin <= end) and cover [lo, hi); counts / offsets / pos_out are host memory.
int search_ranges_host(ThreadCtx &c, const char *text, int64_t n, int64_t nranges, const int64_t *begin, const int64_t *end,
                       int64_t lo, int64_t hi, const char *pat, int32_t m, int64_t *pos_out, int64_t pos_cap, uint64_t *counts,
                       int64_t *offsets);

// K patterns in one pass over device-resident text (bmx_multipat.cu)
bool multi_eligible(int32_t npat, const int32_t *ms);
int multi_scan_resident(ThreadCtx &c, const unsigned char *d_text, int64_t n, int32_t npat, const char *const *pats,
                        const int32_t *ms, int64_t *const *d_out, const int64_t *caps, uint64_t *counts, cudaStream_t st);

// The shared candidate table of a pattern set (bmx_multipat.cu; used by bmx_search_multi and the dictionaries).  One
// gram length q = min(12, m_min - 3) = 4 + q2 + q3 bytes for every pattern and residue.
struct SetHash {
    int32_t m_min = 0, m_max = 0;
    int q2 = 0, q3 = 0;              // bytes the second and third word contribute to a gram
    uint32_t hmul = 0, hmul2 = 0;    // their multipliers (gram_multiplier: the bytes beyond the gram drop out)
};
SetHash set_hash(int32_t npat, const int32_t *ms);
// Hash of the gram that starts at p (host and device alike: the scan hashes aligned text words the same way).
__host__ __device__ inline uint32_t set_gram_hash(const SetHash &sh, const unsigned char *p)
{
    uint32_t w0 = 0u, w1 = 0u, w2 = 0u;
    for (int i = 0; i < 4; ++i) w0 |= (uint32_t)p[i] << (8 * i);
    for (int i = 0; i < sh.q2; ++i) w1 |= (uint32_t)p[4 + i] << (8 * i);
    for (int i = 0; i < sh.q3; ++i) w2 |= (uint32_t)p[8 + i] << (8 * i);
    return w0 + sh.hmul * w1 + sh.hmul2 * w2;
}
// Bytes of the pattern blob: every pattern 16-byte aligned and followed by at least 8 bytes of padding.
size_t set_blob_bytes(int32_t npat, const int32_t *ms);
// Fills bitmap (kMultiBitmapWords words), exact table (2^slots_log2 slots, load <= 1/2), directory and blob, all zeroed
// by the caller: table entry {hash, 0x80000000 | k << 2 | r} for the gram P_k[r .. r+q) of every pattern k and residue r.
void fill_set_tables(int32_t npat, const char *const *pats, const int32_t *ms, const SetHash &sh, int slots_log2, uint32_t *bits,
                     uint2 *table, uint2 *dir, unsigned char *blob);

#ifdef __CUDACC__
// Exclusive prefix of v over a CTA of THREADS threads; *total receives the CTA's sum.  Every thread calls it.
template <int THREADS>
__device__ __forceinline__ unsigned long long cta_exclusive_scan(unsigned long long v, unsigned long long *total)
{
    __shared__ unsigned long long warp_total[THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_total[warp] = x;
    __syncthreads();
    unsigned long long base = 0, sum = 0;
#pragma unroll
    for (int w = 0; w < THREADS / 32; ++w) {
        const unsigned long long t = warp_total[w];
        base += w < warp ? t : 0ull;
        sum += t;
    }
    __syncthreads();   // warp_total may be reused by the next call
    *total = sum;
    return base + x - v;
}
#endif

// Sets the scanner's timing level (bmx_scanner_set_timing) for the scope and restores the caller's level after it.
class ScopedTiming {
public:
    ScopedTiming(bmx_scanner *s, int level) : s_(s), keep_(s->timing_level) { s_->timing_level = level; }
    ~ScopedTiming() { s_->timing_level = keep_; }
    ScopedTiming(const ScopedTiming &) = delete;
    ScopedTiming &operator=(const ScopedTiming &) = delete;

private:
    bmx_scanner *s_;
    int keep_;
};

// Restores the calling thread's current device when the scope ends.
class ScopedDevice {
public:
    ScopedDevice() : have_(cudaGetDevice(&keep_) == cudaSuccess) {}
    ~ScopedDevice()
    {
        if (have_) cudaSetDevice(keep_);
    }
    ScopedDevice(const ScopedDevice &) = delete;
    ScopedDevice &operator=(const ScopedDevice &) = delete;

private:
    int keep_ = 0;
    bool have_;
};

}  // namespace bmx
