// bmx_ranges.cu -- many ranges of one text in one pass: exact per-range counts, CSR offsets and position lists.
//
// Generalises the reference's kernel entry search(text, pattern, se, ans, ...) (kernel1.cl:1, ranges from
// BoyreMoore.cpp:119-141): range d = [begin[d], end[d]) counts the matches lying fully inside it, no halo.  Instead
// of one scan per range the covered bytes are scanned ONCE with positions (the ordinary scan + expand kernels);
// the ascending list L of every match start then answers all ranges at once:
//   rank     a_d = lower_bound(L, begin_d), b_d = lower_bound(L, end_d - m + 1), counts[d] = b_d - a_d; per-CTA
//            sums, and the CTA that arrives last turns them into bases (the scan kernel's own idiom, DESIGN §3.2);
//            device ranges are checked against [0, n] here (range values are only compared, never used as indices)
//   offsets  offsets[d] = CTA base + exclusive scan of the counts inside the CTA; offsets[D] = total
//   gather   out[j] = L[a_d + j - offsets[d]] - begin_d for j < min(total, pos_cap), balanced by output index
// All three run behind the scan on the same stream without waiting for its count: if the count shows that L was
// cut short, the position buffer is grown and everything runs again (the speculation of small_host_search).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>

#include "bmx_ctx.h"

using namespace bmx;

namespace {

constexpr int kRangeThreads = 256;
constexpr int kRangesPerThread = 8;
constexpr int kRangesPerCta = kRangeThreads * kRangesPerThread;   // 2048 ranges per CTA of rank / offsets
constexpr int kGatherThreads = 256;
constexpr int kGatherTile = 2048;    // output positions per CTA step
constexpr int kGatherStage = 4096;   // offsets a tile may span and still search in shared memory (32 KiB)

struct RangeCtrl {                   // device header, zeroed per call; copied to host memory behind the kernels
    unsigned long long bad;          // 1 + index of a range outside [0, n] or with begin > end (0: none)
    unsigned long long total;        // offsets[D]
    unsigned int ticket;             // rank CTAs done
    unsigned int pad[3];
};
constexpr int kCtrlWords = (int)(sizeof(RangeCtrl) / 8);   // int64 slots it takes in the pinned landing area

// first index in [lo, hi) with a[idx] >= key
__device__ __forceinline__ int64_t lower_bound(const int64_t *__restrict__ a, int64_t lo, int64_t hi, int64_t key)
{
    while (lo < hi) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        if (__ldg(a + mid) < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// first index in [lo, hi) with a[idx] > key
__device__ __forceinline__ int64_t upper_bound(const int64_t *a, int64_t lo, int64_t hi, int64_t key)
{
    while (lo < hi) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        if (a[mid] <= key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// Entries of L the scan left: min(count, cap) when the count is on the device, else `cap` itself.
__device__ __forceinline__ int64_t held_entries(const unsigned long long *d_count, int64_t cap)
{
    return d_count ? min((int64_t)*d_count, cap) : cap;
}

__global__ void __launch_bounds__(kRangeThreads) range_rank_kernel(
    const int64_t *__restrict__ L, const unsigned long long *d_count, int64_t L_cap, const int64_t *__restrict__ begin,
    const int64_t *__restrict__ end, int64_t nranges, int64_t n, int32_t m, unsigned long long *__restrict__ counts,
    int64_t *__restrict__ first, unsigned long long *cta_sum, int64_t *offsets, RangeCtrl *ctrl)
{
    const int64_t H = held_entries(d_count, L_cap);
    const int64_t base = (int64_t)blockIdx.x * kRangesPerCta;
    unsigned long long sum = 0;
    for (int k = 0; k < kRangesPerThread; ++k) {
        const int64_t d = base + k * kRangeThreads + threadIdx.x;
        if (d >= nranges) break;
        const int64_t b = begin[d], e = end[d];
        int64_t a = 0, c = 0;
        if (b < 0 || b > e || e > n) {
            atomicMax(&ctrl->bad, (unsigned long long)(d + 1));
        } else {
            a = lower_bound(L, 0, H, b);
            if (e - b >= m) c = lower_bound(L, a, H, e - m + 1) - a;
        }
        counts[d] = (unsigned long long)c;
        first[d] = a;
        sum += (unsigned long long)c;
    }
    unsigned long long cta_total = 0;
    (void)cta_exclusive_scan<kRangeThreads>(sum, &cta_total);
    __shared__ bool last;
    if (threadIdx.x == 0) {
        cta_sum[blockIdx.x] = cta_total;
        __threadfence();
        last = atomicAdd(&ctrl->ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    // the last CTA: per-CTA sums -> exclusive bases, in place; each thread owns a contiguous run of CTAs
    const int64_t G = gridDim.x, per = (G + kRangeThreads - 1) / kRangeThreads;
    const int64_t lo = min(G, (int64_t)threadIdx.x * per), hi = min(G, lo + per);
    unsigned long long local = 0;
    for (int64_t g = lo; g < hi; ++g) local += __ldcg(cta_sum + g);
    unsigned long long total = 0;
    unsigned long long run = cta_exclusive_scan<kRangeThreads>(local, &total);
    for (int64_t g = lo; g < hi; ++g) {
        const unsigned long long v = __ldcg(cta_sum + g);
        cta_sum[g] = run;
        run += v;
    }
    if (threadIdx.x == 0) {
        offsets[nranges] = (int64_t)total;
        ctrl->total = total;
    }
}

__global__ void __launch_bounds__(kRangeThreads) range_offsets_kernel(const unsigned long long *__restrict__ counts,
                                                                       const unsigned long long *__restrict__ cta_base,
                                                                       int64_t nranges, int64_t *__restrict__ offsets)
{
    const int64_t base = (int64_t)blockIdx.x * kRangesPerCta + (int64_t)threadIdx.x * kRangesPerThread;
    unsigned long long c[kRangesPerThread];
    unsigned long long local = 0;
#pragma unroll
    for (int k = 0; k < kRangesPerThread; ++k) {
        c[k] = base + k < nranges ? counts[base + k] : 0ull;
        local += c[k];
    }
    unsigned long long cta_total = 0;
    unsigned long long run = cta_base[blockIdx.x] + cta_exclusive_scan<kRangeThreads>(local, &cta_total);
#pragma unroll
    for (int k = 0; k < kRangesPerThread; ++k) {
        if (base + k < nranges) offsets[base + k] = (int64_t)run;
        run += c[k];
    }
}

// Work is split by output index: a CTA takes kGatherTile consecutive outputs, finds the ranges they belong to with
// two binary searches over offsets and stages those ranges' offsets in shared memory, so one range of 10^8 hits and
// 10^7 ranges of one hit each cost the same per output.
__global__ void __launch_bounds__(kGatherThreads) range_gather_kernel(
    const int64_t *__restrict__ L, const int64_t *__restrict__ begin, const int64_t *__restrict__ first,
    const int64_t *__restrict__ offsets, int64_t nranges, int64_t pos_cap, int64_t *__restrict__ out)
{
    __shared__ int64_t s_off[kGatherStage];
    __shared__ int64_t s_d0, s_d1;
    const int64_t nout = min(offsets[nranges], pos_cap);
    for (int64_t j0 = (int64_t)blockIdx.x * kGatherTile; j0 < nout; j0 += (int64_t)gridDim.x * kGatherTile) {
        const int64_t j1 = min(nout, j0 + kGatherTile);
        if (threadIdx.x == 0) {
            // the range holding output j is the last d with offsets[d] <= j (empty ranges in front of it share its offset)
            const int64_t d0 = upper_bound(offsets, 0, nranges + 1, j0) - 1;
            s_d0 = d0;
            s_d1 = upper_bound(offsets, d0, nranges + 1, j1 - 1) - 1;
        }
        __syncthreads();
        const int64_t d0 = s_d0, span = s_d1 - d0 + 1;
        const bool staged = span <= kGatherStage;
        if (staged)
            for (int64_t i = threadIdx.x; i < span; i += kGatherThreads) s_off[i] = offsets[d0 + i];
        __syncthreads();
        const int64_t *off = staged ? s_off : offsets + d0;
        for (int64_t j = j0 + threadIdx.x; j < j1; j += kGatherThreads) {
            const int64_t i = upper_bound(off, 0, span, j) - 1;
            const int64_t d = d0 + i;
            out[j] = __ldg(L + first[d] + (j - off[i])) - begin[d];
        }
        __syncthreads();   // s_off and s_d0 are rewritten by the next tile
    }
}

int sm_count()
{
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
        (void)cudaGetLastError();
        sms = 148;
    }
    return sms;
}

int ensure_landing(ThreadCtx &c)
{
    if (!c.h_small) BMX_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&c.h_small), (size_t)kSmallSpec * 8, cudaHostAllocDefault));
    return BMX_OK;
}

// Enqueues rank, offsets and (d_pos && pos_cap > 0) gather on `st` over the list L (held entries: see held_entries),
// then copies the RangeCtrl header to c.h_small.  Scratch: c.misc.  Nothing waits for the device.
int launch_ranges(ThreadCtx &c, const int64_t *L, const unsigned long long *d_count, int64_t L_cap, int64_t nranges,
                  const int64_t *d_begin, const int64_t *d_end, int64_t n, int32_t m, int64_t *d_pos, int64_t pos_cap,
                  uint64_t *d_counts, int64_t *d_offsets, cudaStream_t st)
{
    const int64_t G = (nranges + kRangesPerCta - 1) / kRangesPerCta;
    const size_t off_sum = 256, off_first = off_sum + (((size_t)G * 8 + 255) & ~size_t(255));
    if (int rc = ensure_buf(c, c.misc, off_first + (size_t)nranges * 8)) return rc;
    unsigned char *scratch = static_cast<unsigned char *>(c.misc.p);
    RangeCtrl *ctrl = reinterpret_cast<RangeCtrl *>(scratch);
    unsigned long long *cta_sum = reinterpret_cast<unsigned long long *>(scratch + off_sum);
    int64_t *first = reinterpret_cast<int64_t *>(scratch + off_first);
    BMX_CUDA(cudaMemsetAsync(ctrl, 0, sizeof(RangeCtrl), st));
    range_rank_kernel<<<(unsigned)G, kRangeThreads, 0, st>>>(L, d_count, L_cap, d_begin, d_end, nranges, n, m,
                                                             reinterpret_cast<unsigned long long *>(d_counts), first, cta_sum,
                                                             d_offsets, ctrl);
    range_offsets_kernel<<<(unsigned)G, kRangeThreads, 0, st>>>(reinterpret_cast<const unsigned long long *>(d_counts), cta_sum,
                                                                nranges, d_offsets);
    if (d_pos && pos_cap > 0) {
        const int64_t tiles = (pos_cap + kGatherTile - 1) / kGatherTile;
        const unsigned grid = (unsigned)std::min<int64_t>(tiles, (int64_t)sm_count() * 4);
        range_gather_kernel<<<grid, kGatherThreads, 0, st>>>(L, d_begin, first, d_offsets, nranges, pos_cap, d_pos);
    }
    if (cudaError_t e = cudaGetLastError(); e != cudaSuccess) return fail(BMX_E_CUDA, "range kernels: %s", cudaGetErrorString(e));
    BMX_CUDA(cudaMemcpyAsync(c.h_small, ctrl, sizeof(RangeCtrl), cudaMemcpyDeviceToHost, st));
    return BMX_OK;
}

RangeCtrl landed(const ThreadCtx &c)
{
    RangeCtrl r;
    memcpy(&r, c.h_small, sizeof r);
    return r;
}

// Checks a host range set: every range inside [0, n] with begin <= end.  *lo / *hi: the covered bytes.
int check_host_ranges(int64_t n, int64_t nranges, const int64_t *begin, const int64_t *end, int64_t *lo, int64_t *hi, const char *who)
{
    *lo = n;
    *hi = 0;
    for (int64_t d = 0; d < nranges; ++d) {
        if (begin[d] < 0 || begin[d] > end[d] || end[d] > n)
            return fail(BMX_E_BADARG, "%s: range %lld = [%lld, %lld) is not inside [0, %lld] with begin <= end", who, (long long)d,
                        (long long)begin[d], (long long)end[d], (long long)n);
        *lo = std::min(*lo, begin[d]);
        *hi = std::max(*hi, end[d]);
    }
    if (*lo > *hi) *lo = *hi;
    return BMX_OK;
}

}  // namespace

namespace bmx {

// Host text and ranges (already checked) -> host outputs.  The covered bytes [lo, hi) go through the ordinary chunked
// ingest with positions (L holds absolute starts, pos_base = lo); the range kernels run on the resulting list.
int search_ranges_host(ThreadCtx &c, const char *text, int64_t n, int64_t nranges, const int64_t *begin, const int64_t *end,
                       int64_t lo, int64_t hi, const char *pat, int32_t m, int64_t *pos_out, int64_t pos_cap, uint64_t *counts,
                       int64_t *offsets)
{
    if (int rc = ensure_streams(c, 0)) return rc;
    if (int rc = ensure_landing(c)) return rc;
    ScopedTiming timing(c.scanner, 0);
    const int64_t span = hi - lo;
    int64_t held = 0;
    if (span >= m) {
        uint64_t count = 0;
        int64_t dev_cap = 0;
        if (int rc = ingest_shard(c, c.device, text + lo, span, pat, m, lo, span - m + 1, &count, &dev_cap)) return rc;
        held = std::min<int64_t>((int64_t)count, dev_cap);
    }
    if (!pos_out) pos_cap = 0;
    cudaStream_t st = c.scan_stream;
    // device copies of the ranges and the outputs: [begin | end | counts | offsets | positions]
    const size_t rbytes = ((size_t)nranges * 8 + 255) & ~size_t(255), obytes = ((size_t)(nranges + 1) * 8 + 255) & ~size_t(255);
    int64_t gcap = std::min<int64_t>(pos_cap, std::max<int64_t>(held, kSmallSpec));   // first guess: one output per hit
    const int64_t spec = kSmallSpec - kCtrlWords;                                      // outputs read back with the header
    for (int pass = 0; pass < 2; ++pass) {
        if (int rc = ensure_buf(c, c.aux, 3 * rbytes + obytes + (size_t)gcap * 8)) return rc;
        unsigned char *a = static_cast<unsigned char *>(c.aux.p);
        int64_t *d_begin = reinterpret_cast<int64_t *>(a), *d_end = reinterpret_cast<int64_t *>(a + rbytes);
        uint64_t *d_counts = reinterpret_cast<uint64_t *>(a + 2 * rbytes);
        int64_t *d_offsets = reinterpret_cast<int64_t *>(a + 3 * rbytes);
        int64_t *d_pos = reinterpret_cast<int64_t *>(a + 3 * rbytes + obytes);
        BMX_CUDA(cudaMemcpyAsync(d_begin, begin, (size_t)nranges * 8, cudaMemcpyHostToDevice, st));
        BMX_CUDA(cudaMemcpyAsync(d_end, end, (size_t)nranges * 8, cudaMemcpyHostToDevice, st));
        if (int rc = launch_ranges(c, static_cast<const int64_t *>(c.pos.p), nullptr, held, nranges, d_begin, d_end, n, m,
                                   gcap > 0 ? d_pos : nullptr, gcap, d_counts, d_offsets, st))
            return rc;
        if (gcap > 0) BMX_CUDA(cudaMemcpyAsync(c.h_small + kCtrlWords, d_pos, (size_t)std::min(gcap, spec) * 8, cudaMemcpyDeviceToHost, st));
        BMX_CUDA(cudaMemcpyAsync(counts, d_counts, (size_t)nranges * 8, cudaMemcpyDeviceToHost, st));
        BMX_CUDA(cudaMemcpyAsync(offsets, d_offsets, (size_t)(nranges + 1) * 8, cudaMemcpyDeviceToHost, st));
        BMX_CUDA(cudaStreamSynchronize(st));
        const RangeCtrl r = landed(c);
        if (r.bad) return fail(BMX_E_BADARG, "range %lld outside [0, %lld]", (long long)(r.bad - 1), (long long)n);
        const int64_t nout = std::min<int64_t>((int64_t)r.total, pos_cap);
        if (nout > gcap) {   // overlapping ranges hold more outputs than the list has hits: gather again with room for them
            gcap = nout;
            continue;
        }
        if (nout > 0) {
            memcpy(pos_out, c.h_small + kCtrlWords, (size_t)std::min(nout, spec) * 8);
            if (nout > spec) {
                BMX_CUDA(cudaMemcpyAsync(pos_out + spec, d_pos + spec, (size_t)(nout - spec) * 8, cudaMemcpyDeviceToHost, st));
                BMX_CUDA(cudaStreamSynchronize(st));
            }
        }
        return BMX_OK;
    }
    return fail(BMX_E_CUDA, "bmx_search_ranges: position buffer did not converge");
}

}  // namespace bmx

extern "C" {

int bmx_search_ranges(int device, const char *text, int64_t n, int64_t nranges, const int64_t *begin, const int64_t *end,
                      const char *pat, int32_t m, int64_t *pos_out, int64_t pos_cap, uint64_t *counts, int64_t *offsets)
{
    if (!pat || !offsets || nranges < 0 || (nranges > 0 && (!begin || !end || !counts)))
        return fail(BMX_E_BADARG, "bmx_search_ranges: NULL argument or nranges < 0");
    if (int rc = check_text(text, n, "bmx_search_ranges")) return rc;
    if (pos_cap < 0) return fail(BMX_E_BADARG, "bmx_search_ranges: pos_cap < 0");
    if (int rc = check_pattern(m)) return rc;
    int64_t lo = 0, hi = 0;
    if (int rc = check_host_ranges(n, nranges, begin, end, &lo, &hi, "bmx_search_ranges")) return rc;
    ThreadCtx *c = nullptr;
    if (int rc = get_ctx(device, &c)) return rc;
    offsets[0] = 0;
    if (nranges == 0) return BMX_OK;
    return search_ranges_host(*c, text, n, nranges, begin, end, lo, hi, pat, m, pos_out, pos_cap, counts, offsets);
}

int bmx_search_ranges_device(const void *d_text, int64_t n, int64_t nranges, const int64_t *d_begin, const int64_t *d_end,
                             const char *pat, int32_t m, int64_t *d_pos_out, int64_t pos_cap, uint64_t *d_counts,
                             int64_t *d_offsets, uint64_t *total_out, void *stream)
{
    if (!pat || !d_offsets || !total_out || nranges < 0 || (nranges > 0 && (!d_begin || !d_end || !d_counts)))
        return fail(BMX_E_BADARG, "bmx_search_ranges_device: NULL argument or nranges < 0");
    if (int rc = check_text(d_text, n, "bmx_search_ranges_device")) return rc;
    if (pos_cap < 0) return fail(BMX_E_BADARG, "bmx_search_ranges_device: pos_cap < 0");
    if (int rc = check_pattern(m)) return rc;
    *total_out = 0;
    ThreadCtx *c = nullptr;
    if (int rc = current_ctx(&c)) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (nranges == 0) {
        BMX_CUDA(cudaMemsetAsync(d_offsets, 0, 8, st));
        BMX_CUDA(cudaStreamSynchronize(st));
        return BMX_OK;
    }
    if (int rc = ensure_landing(*c)) return rc;
    if (!d_pos_out) pos_cap = 0;
    bmx_scanner *s = c->scanner;
    ScopedTiming timing(s, 0);
    // L over the whole text, first guess one hit per 64 bytes; the range kernels follow the scan without a wait
    const int64_t want = n >= m ? n - m + 1 : 0;
    int64_t cap = want > 0 ? first_pos_room(*c, n, m, want) : 0;
    for (int pass = 0; pass < 2; ++pass) {
        if (cap > 0)
            if (int rc = ensure_buf(*c, c->pos, (size_t)cap * 8)) return rc;
        int64_t *L = static_cast<int64_t *>(c->pos.p);
        const unsigned long long *d_count = nullptr;
        if (want > 0) {
            int rc = bmx_scanner_set_pattern(s, pat, m, BMX_VARIANT_AUTO, st);
            if (rc == BMX_OK) rc = bmx_scanner_begin(s, L, cap, st);
            if (rc == BMX_OK) rc = bmx_scanner_scan(s, d_text, n, 0, st);
            if (rc != BMX_OK) return rc;
            d_count = result_slot(s);
        }
        if (int rc = launch_ranges(*c, L, d_count, cap, nranges, d_begin, d_end, n, m, d_pos_out, pos_cap, d_counts, d_offsets, st))
            return rc;
        uint64_t count = 0;
        if (want > 0) {
            if (int rc = bmx_scanner_finish(s, &count, nullptr, st)) return rc;   // the one synchronisation
        } else {
            BMX_CUDA(cudaStreamSynchronize(st));
        }
        if ((int64_t)count > cap) {   // denser than the guess: L was cut short, so every range result is redone
            cap = (int64_t)count;
            continue;
        }
        const RangeCtrl r = landed(*c);
        if (r.bad)
            return fail(BMX_E_BADARG, "bmx_search_ranges_device: range %lld is not inside [0, %lld] with begin <= end",
                        (long long)(r.bad - 1), (long long)n);
        *total_out = r.total;
        return BMX_OK;
    }
    return fail(BMX_E_CUDA, "bmx_search_ranges_device: position buffer did not converge");
}

}  // extern "C"
