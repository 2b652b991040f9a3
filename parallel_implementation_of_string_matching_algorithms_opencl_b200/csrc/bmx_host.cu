// bmx_host.cu -- the host-pointer entry points of libbmx.so: text in host memory -> hits in host memory.
//
// Replaces the reference's buffer set and blocking transfers, BoyreMoore/BoyreMoore/BoyreMoore.cpp:233-252
// (clCreateBuffer x6, clEnqueueWriteBuffer x5 with CL_TRUE) and the read-back :283-286.  The reference copies
// the whole text in one blocking call and only then launches; here the text crosses PCIe in chunks on a copy
// stream while the scan stream scans everything that has already arrived.
//
// Two layouts of the device copy:
//   resident  the text fits: one cached buffer of n bytes, chunk k is scanned together with the (m-1) bytes in
//             front of it (matches straddling chunk seams are found exactly once, the list stays ascending); the
//             copy stays available (bmx_search_multi; growing the position buffer after a dense first pass).
//   ring      the text is larger than the device can hold (or BMX_RESIDENT_MAX_MB says so): four chunk slots,
//             each with room for the previous chunk's last (m-1) bytes in front; chunk k+4 overwrites chunk k once
//             its scan is done.  Device memory is constant in n.
// The position buffer is never sized by the worst case (8 bytes per text byte): it starts at max(1 Mi, n/64)
// entries and is grown to the true count only when a text turns out to be denser than that (the resident copy is
// then simply re-scanned; a ring text is ingested once more).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "bmx_ctx.h"

using namespace bmx;

namespace {

constexpr int kRing = 4;

// memcpy split over a few host threads: one core moves ~10 GB/s, a PCIe Gen5 x16 link takes ~55 GB/s
void parallel_copy(void *dst, const void *src, size_t bytes, int threads)
{
    if (threads <= 1 || bytes < (size_t(8) << 20)) {
        memcpy(dst, src, bytes);
        return;
    }
    const size_t slice = ((bytes / (size_t)threads) + 4095) & ~size_t(4095);
    std::vector<std::thread> helpers;
    for (int t = 1; t < threads; ++t) {
        const size_t lo = std::min(bytes, slice * (size_t)t), hi = std::min(bytes, lo + slice);
        if (hi > lo)
            helpers.emplace_back([=] { memcpy(static_cast<char *>(dst) + lo, static_cast<const char *>(src) + lo, hi - lo); });
    }
    memcpy(dst, src, std::min(bytes, slice));
    for (auto &h : helpers) h.join();
}

bool is_pinned_host(const void *p)
{
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeHost;
}

// One search over device-resident text with a position buffer that follows the count: first pass with the
// cached buffer, and only if the text holds more hits than it has room for (and the caller wants them) a
// second pass with a buffer of the right size.  On return ctx.pos holds min(count, *dev_cap) positions.
int scan_resident(ThreadCtx &c, const unsigned char *d_text, int64_t n, const char *pat, int32_t m, int32_t variant,
                  int64_t pos_base, int64_t want_cap, uint64_t *count, int64_t *dev_cap, bmx_stats *stats)
{
    int64_t cap = first_pos_room(c, n, m, want_cap);
    for (int pass = 0; pass < 2; ++pass) {
        if (cap > 0)
            if (int rc = ensure_buf(c, c.pos, (size_t)cap * 8)) return rc;
        if (int rc = search_once(c.scanner, pat, m, variant, d_text, n, pos_base, cap > 0 ? static_cast<int64_t *>(c.pos.p) : nullptr,
                                 cap, count, stats, c.scan_stream))
            return rc;
        const int64_t need = std::min<int64_t>(want_cap, (int64_t)*count);
        if (need <= cap) break;
        cap = need;
    }
    *dev_cap = cap;
    return BMX_OK;
}

// Small host texts -- the reference's own fixtures are 60 B .. 560 KB (BoyreMoore/**/input*.txt) and its timed window
// is one launch plus an 8-byte read (BoyreMoore.cpp:258-290) -- are latency, not bandwidth: everything goes through ONE
// stream (no copy stream, no events, no pinned-memory query), and the first kSmallSpec positions travel back to a pinned
// landing area right behind the kernels, so that the call synchronises once instead of twice (count, then positions).
// Falls back to the resident re-scan when the text holds more hits than the position buffer (scan_resident).
constexpr int64_t kSmallHostBytes = int64_t(4) << 20;
int small_host_search(ThreadCtx &c, const char *text, int64_t n, const char *pat, int32_t m, int32_t variant,
                      int64_t *pos_out, int64_t want_cap, uint64_t *count_out, bmx_stats *stats)
{
    if (int rc = ensure_streams(c, 0)) return rc;
    if (int rc = ensure_buf(c, c.text, (size_t)n + 16)) return rc;
    const int64_t cap = first_pos_room(c, n, m, want_cap);
    if (cap > 0)
        if (int rc = ensure_buf(c, c.pos, (size_t)cap * 8)) return rc;
    if (cap > 0 && !c.h_small) BMX_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&c.h_small), (size_t)kSmallSpec * 8, cudaHostAllocDefault));
    cudaStream_t st = c.scan_stream;
    unsigned char *d_text = static_cast<unsigned char *>(c.text.p);
    // (a pageable source is staged by the runtime before the call returns: the caller's buffer is free afterwards)
    BMX_CUDA(cudaMemcpyAsync(d_text, text, (size_t)n, cudaMemcpyHostToDevice, st));
    int rc = bmx_scanner_set_pattern(c.scanner, pat, m, variant, st);
    if (rc == BMX_OK) rc = bmx_scanner_begin(c.scanner, cap > 0 ? static_cast<int64_t *>(c.pos.p) : nullptr, cap, st);
    if (rc == BMX_OK) rc = bmx_scanner_scan(c.scanner, d_text, n, 0, st);
    if (rc != BMX_OK) return rc;
    const int64_t spec = std::min<int64_t>(cap, kSmallSpec);
    if (spec > 0) BMX_CUDA(cudaMemcpyAsync(c.h_small, c.pos.p, (size_t)spec * 8, cudaMemcpyDeviceToHost, st));
    uint64_t count = 0;
    if ((rc = bmx_scanner_finish(c.scanner, &count, stats, st)) != BMX_OK) return rc;   // the one synchronisation
    *count_out = count;
    int64_t dev_cap = cap;
    const int64_t need = std::min<int64_t>(want_cap, (int64_t)count);
    if (need > cap) {   // denser than the buffer: the text is resident, scan it again with room for what the caller asked for
        if ((rc = scan_resident(c, d_text, n, pat, m, variant, 0, want_cap, &count, &dev_cap, stats)) != BMX_OK) return rc;
        *count_out = count;
        BMX_CUDA(cudaMemcpyAsync(pos_out, c.pos.p, (size_t)std::min<int64_t>({(int64_t)count, dev_cap, want_cap}) * 8, cudaMemcpyDeviceToHost, st));
        BMX_CUDA(cudaStreamSynchronize(st));
        return BMX_OK;
    }
    if (need > 0) {
        memcpy(pos_out, c.h_small, (size_t)std::min(need, spec) * 8);
        if (need > spec) {
            BMX_CUDA(cudaMemcpyAsync(pos_out + spec, static_cast<int64_t *>(c.pos.p) + spec, (size_t)(need - spec) * 8, cudaMemcpyDeviceToHost, st));
            BMX_CUDA(cudaStreamSynchronize(st));
        }
    }
    return BMX_OK;
}

struct Ingest {
    // in
    int64_t want_cap = 0;        // positions the caller can use (0: count only)
    bool find_first = false;     // stop copying and scanning behind the first match
    bool copy_only = false;      // ingest without scanning into the resident layout: the caller scans the device copy
                                 // itself (bmx_search_multi); NOMEM when the text does not fit
    // out
    uint64_t count = 0;
    int64_t dev_cap = 0;         // ctx.pos holds min(count, dev_cap) positions
    int64_t first = -1;          // find_first: smallest start position or -1
    bool resident = false;       // ctx.text holds the whole text
    bmx_stats stats{};
};

// Host text -> device (chunked, overlapped with scanning) -> hits in ctx.pos.
int ingest_and_scan(ThreadCtx &ctx, int device, const char *text, int64_t n, const char *pat, int32_t m, int64_t pos_base,
                    int32_t variant, Ingest *io)
{
    ThreadCtx *c = &ctx;
    io->count = 0;
    io->dev_cap = 0;
    io->first = -1;
    io->resident = false;
    io->stats = bmx_stats{};
    if (n < m && !(io->copy_only && n > 0)) return BMX_OK;
    BMX_CUDA(cudaSetDevice(device));

    int64_t chunk = (int64_t)std::max(1, env_int("BMX_H2D_CHUNK_MB", 64)) << 20;
    if (const int kb = env_int("BMX_H2D_CHUNK_KB", 0)) chunk = (int64_t)kb << 10;   // test knob: many tiny chunks
    chunk = (std::max<int64_t>(chunk, (int64_t)m * 2) + 15) & ~int64_t(15);
    const int64_t nchunks = (n + chunk - 1) / chunk;
    // events: [0] copy of chunk k done, [1 .. kBounce] bounce buffer free, [1+kBounce .. +kRing) ring slot free,
    // then two "find-first result of scan q is in host memory" events.  An event is re-recorded freely: a stream
    // wait captures the record that precedes it.
    const size_t ev_copy = 0, ev_bounce = 1, ev_slot = 1 + kBounce, ev_find = 1 + kBounce + kRing;
    if (int rc = ensure_streams(*c, ev_find + 2)) return rc;
    // work of an earlier call on these streams may still use the cached buffers
    const int64_t carry = m - 1;
    const size_t pre = ((size_t)carry + 15 + 16) & ~size_t(15);

    // ---- layout of the device copy
    const int limit_mb = env_int("BMX_RESIDENT_MAX_MB", -1);
    const size_t resident_need = (size_t)n + 16;
    bool resident;
    if (limit_mb >= 0) {
        resident = resident_need <= ((size_t)limit_mb << 20);
    } else if (resident_need <= c->text.cap) {
        resident = true;   // fits the buffer we already own (the common case of repeated calls): no query
    } else {
        // the scan's own scratch takes ~n/8 bytes and the positions a little: leave a quarter of what is free alone
        size_t free_b = 0, total_b = 0;
        BMX_CUDA(cudaMemGetInfo(&free_b, &total_b));
        resident = resident_need <= (size_t)((double)(free_b + c->text.cap) * 0.75);
    }
    if (resident && ensure_buf(*c, c->text, resident_need) != BMX_OK) resident = false;   // fragmentation etc.: stream it
    if (!resident) {
        if (io->copy_only) return fail(BMX_E_NOMEM, "text of %lld bytes does not fit on the device", (long long)n);
        const size_t slot_stride = pre + (size_t)chunk + 16;
        if (int rc = ensure_buf(*c, c->text, slot_stride * kRing)) return rc;
    }
    const size_t slot_stride = pre + (size_t)chunk + 16;
    unsigned char *d_text = static_cast<unsigned char *>(c->text.p);
    io->resident = resident;

    const bool pinned = is_pinned_host(text);
    int staging_threads = env_int("BMX_STAGING_THREADS", 16);  // host threads filling a bounce buffer: 8 -> 39.9, 16 -> 42.8, 32 -> 43.2 GB/s (profiles/e2e_host_memory_r02.txt)
    staging_threads = (int)std::max(1u, std::min<unsigned>((unsigned)std::max(1, std::min(64, staging_threads)), std::thread::hardware_concurrency()));
    if (!pinned && c->bounce_bytes < (size_t)std::min(chunk, n)) {
        for (int b = 0; b < kBounce; ++b) {
            if (c->bounce[b]) cudaFreeHost(c->bounce[b]);
            c->bounce[b] = nullptr;
        }
        c->bounce_bytes = 0;
        for (int b = 0; b < kBounce; ++b) BMX_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&c->bounce[b]), (size_t)std::min(chunk, n), cudaHostAllocDefault));
        c->bounce_bytes = (size_t)std::min(chunk, n);
    }

    int64_t cap = io->find_first ? 0 : first_pos_room(*c, n, m, io->want_cap);
    for (int pass = 0; pass < 2; ++pass) {
        if (cap > 0)
            if (int rc = ensure_buf(*c, c->pos, (size_t)cap * 8)) return rc;
        if (pass == 1 && resident) {
            // the text is already on the device: one scan with a buffer that has room for what the caller wants
            uint64_t count = 0;
            int64_t dev_cap = 0;
            if (int rc = scan_resident(*c, d_text, n, pat, m, variant, pos_base, io->want_cap, &count, &dev_cap, &io->stats)) return rc;
            io->count = count;
            io->dev_cap = dev_cap;
            return BMX_OK;
        }
        // the copy stream must not overwrite text that scans of an earlier call (or pass) still read
        BMX_CUDA(cudaEventRecord(c->events[ev_copy], c->scan_stream));
        BMX_CUDA(cudaStreamWaitEvent(c->copy_stream, c->events[ev_copy], 0));
        int rc = BMX_OK;
        if (!io->copy_only) {
            rc = bmx_scanner_set_pattern(c->scanner, pat, m, variant, c->scan_stream);
            if (rc == BMX_OK)
                rc = io->find_first ? scanner_begin_find(c->scanner, c->scan_stream)
                                    : bmx_scanner_begin(c->scanner, cap > 0 ? static_cast<int64_t *>(c->pos.p) : nullptr, cap, c->scan_stream);
            if (rc != BMX_OK) return rc;
        }

        int64_t scanned = 0;  // resident layout: start positions < scanned are done
        int64_t q = 0;        // find-first: scans enqueued so far
        bool found = false;
        volatile unsigned long long *h_first = c->scanner->h_result + 1;
        auto first_of = [&](int64_t qq) -> bool {   // waits for scan qq; its last CTA left the best match so far in host memory
            if (cudaEventSynchronize(c->events[ev_find + (size_t)(qq & 1)]) != cudaSuccess) return false;
            const long long f = (long long)*h_first;
            if (f < 0) return false;
            io->first = (int64_t)f;
            return true;
        };
        unsigned char *prev_dst = nullptr;
        int64_t prev_len = 0;
        for (int64_t k = 0; k < nchunks && !found; ++k) {
            const int64_t off = k * chunk;
            const int64_t len = std::min(chunk, n - off);
            unsigned char *dst = resident ? d_text + off : d_text + (size_t)(k % kRing) * slot_stride + pre;
            if (!resident && k >= kRing)   // slot reuse: chunk k-kRing and the seam copy that read its tail are scanned once scan k-kRing+1 is done
                BMX_CUDA(cudaStreamWaitEvent(c->copy_stream, c->events[ev_slot + (size_t)((k + 1) % kRing)], 0));
            const char *src = text + off;
            if (!pinned) {
                const int b = (int)(k % kBounce);
                // the bounce buffer is free once the copy that used it kBounce chunks ago has finished
                if (k >= kBounce) BMX_CUDA(cudaEventSynchronize(c->events[ev_bounce + (size_t)b]));
                parallel_copy(c->bounce[b], src, (size_t)len, staging_threads);
                BMX_CUDA(cudaMemcpyAsync(dst, c->bounce[b], (size_t)len, cudaMemcpyHostToDevice, c->copy_stream));
                BMX_CUDA(cudaEventRecord(c->events[ev_bounce + (size_t)b], c->copy_stream));
            } else {
                BMX_CUDA(cudaMemcpyAsync(dst, src, (size_t)len, cudaMemcpyHostToDevice, c->copy_stream));
            }
            BMX_CUDA(cudaEventRecord(c->events[ev_copy], c->copy_stream));
            BMX_CUDA(cudaStreamWaitEvent(c->scan_stream, c->events[ev_copy], 0));
            bool scanned_now = false;
            if (resident) {
                // every match lying fully inside the bytes copied so far, not yet reported
                const int64_t have = off + len, span = have - scanned;
                if (span >= m && !io->copy_only) {
                    if ((rc = bmx_scanner_scan(c->scanner, d_text + scanned, span, pos_base + scanned, c->scan_stream)) != BMX_OK) return rc;
                    scanned = have - m + 1;
                    scanned_now = true;
                }
            } else {
                // the previous chunk's last m-1 bytes go in front of this one (device to device, a few bytes)
                const int64_t tail = k == 0 ? 0 : std::min<int64_t>(carry, prev_len);
                if (tail > 0) BMX_CUDA(cudaMemcpyAsync(dst - tail, prev_dst + prev_len - tail, (size_t)tail, cudaMemcpyDeviceToDevice, c->scan_stream));
                if (tail + len >= m) {
                    if ((rc = bmx_scanner_scan(c->scanner, dst - tail, tail + len, pos_base + off - tail, c->scan_stream)) != BMX_OK) return rc;
                    scanned_now = true;
                }
                BMX_CUDA(cudaEventRecord(c->events[ev_slot + (size_t)(k % kRing)], c->scan_stream));
                prev_dst = dst;
                prev_len = len;
            }
            if (io->find_first && scanned_now) {
                BMX_CUDA(cudaEventRecord(c->events[ev_find + (size_t)(q & 1)], c->scan_stream));
                if (q >= 1) found = first_of(q - 1);   // one scan behind: the GPU never waits for the host
                ++q;
            }
        }
        if (io->copy_only) {
            BMX_CUDA(cudaStreamSynchronize(c->scan_stream));   // every chunk has landed (the scan stream waited for each copy)
            return BMX_OK;
        }
        uint64_t count = 0;
        if ((rc = bmx_scanner_finish(c->scanner, &count, &io->stats, c->scan_stream)) != BMX_OK) return rc;
        if (io->find_first) {
            if (!found && q >= 1) first_of(q - 1);
            // copies of chunks behind the match may still be in flight: the caller's buffer must be free on return
            BMX_CUDA(cudaStreamSynchronize(c->copy_stream));
            return BMX_OK;
        }
        io->count = count;
        io->dev_cap = cap;
        const int64_t need = std::min<int64_t>(io->want_cap, (int64_t)count);
        if (need <= cap) break;
        cap = need;   // denser than one hit per 64 bytes: go again with room for what the caller asked for
    }
    return BMX_OK;
}

}  // namespace

namespace bmx {
int ingest_shard(ThreadCtx &ctx, int device, const char *text, int64_t n, const char *pat, int32_t m, int64_t pos_base,
                 int64_t want_cap, uint64_t *count, int64_t *dev_cap)
{
    Ingest io;
    io.want_cap = want_cap;
    const int rc = ingest_and_scan(ctx, device, text, n, pat, m, pos_base, BMX_VARIANT_AUTO, &io);
    *count = io.count;
    *dev_cap = io.dev_cap;
    return rc;
}

int copy_text_resident(ThreadCtx &ctx, const char *text, int64_t n)
{
    Ingest io;
    io.copy_only = true;
    return ingest_and_scan(ctx, ctx.device, text, n, "", 1, 0, BMX_VARIANT_AUTO, &io);   // (a copy reads no pattern)
}
}  // namespace bmx

extern "C" {

int bmx_search_ex(int device, const char *text, int64_t n, const char *pat, int32_t m, int64_t *pos_out,
                  int64_t pos_cap, uint64_t *count_out, int32_t variant, bmx_stats *stats)
{
    if (!count_out || !pat) return fail(BMX_E_BADARG, "bmx_search: pat/count_out must be non-NULL");
    if (int rc = check_text(text, n, "bmx_search")) return rc;
    if (pos_cap < 0) return fail(BMX_E_BADARG, "pos_cap < 0");
    if (int rc = check_pattern(m)) return rc;
    ThreadCtx *c = nullptr;
    if (int rc = get_ctx(device, &c)) return rc;
    *count_out = 0;
    if (stats) *stats = bmx_stats{};
    if (n < m) return BMX_OK;
    // CUDA-event instrumentation only when the caller asks for the times: the records cost ~15 us per call
    // (profiles/call_latency_r02.txt), which is nothing for 4 GiB and a fifth of a call on the reference's 500 KB fixture
    ScopedTiming timing(c->scanner, stats ? 2 : 0);
    if (n <= kSmallHostBytes && env_int("BMX_SMALL_HOST", 1) != 0 && env_int("BMX_RESIDENT_MAX_MB", -1) < 0 && env_int("BMX_H2D_CHUNK_KB", 0) == 0)
        return small_host_search(*c, text, n, pat, m, variant, pos_out, pos_out ? std::min(pos_cap, n - m + 1) : 0, count_out, stats);
    Ingest io;
    io.want_cap = pos_out ? std::min(pos_cap, n - m + 1) : 0;
    if (int rc = ingest_and_scan(*c, device, text, n, pat, m, 0, variant, &io)) return rc;
    *count_out = io.count;
    if (stats) *stats = io.stats;
    const int64_t ncopy = std::min<int64_t>({(int64_t)io.count, io.dev_cap, io.want_cap});
    if (ncopy > 0) BMX_CUDA(cudaMemcpyAsync(pos_out, c->pos.p, (size_t)ncopy * 8, cudaMemcpyDeviceToHost, c->scan_stream));
    BMX_CUDA(cudaStreamSynchronize(c->scan_stream));
    return BMX_OK;
}

int bmx_search(const char *text, int64_t n, const char *pat, int32_t m, int64_t *pos_out, int64_t pos_cap,
               uint64_t *count_out)
{
    ThreadCtx *c = nullptr;
    if (int rc = current_ctx(&c)) return rc;
    return bmx_search_ex(c->device, text, n, pat, m, pos_out, pos_cap, count_out, BMX_VARIANT_AUTO, nullptr);
}

// K patterns over one host text: the text crosses PCIe ONCE (chunked, overlapped with the first scan); after
// that all K patterns are searched in the resident copy -- in one pass over the text when the patterns allow
// it (bmx_multi_scan.cu: shared candidate table), else pattern by pattern.
int bmx_search_multi(int device, const char *text, int64_t n, int32_t npat, const char *const *pats, const int32_t *ms,
                     int64_t *const *pos_out, const int64_t *pos_cap, uint64_t *counts)
{
    if (int rc = check_text(text, n, "bmx_search_multi")) return rc;
    if (int rc = check_pattern_set(npat, pats, ms, pos_out, pos_cap, counts, "bmx_search_multi")) return rc;
    ThreadCtx *c = nullptr;
    if (int rc = get_ctx(device, &c)) return rc;
    if (npat == 0 || n == 0) return BMX_OK;
    auto cap_of = [&](int32_t k) -> int64_t {
        if (!pos_out || !pos_out[k] || n < ms[k]) return 0;
        return std::min(pos_cap[k], n - ms[k] + 1);
    };
    auto fetch = [&](int32_t k, uint64_t count, int64_t dev_cap) -> int {
        const int64_t ncopy = std::min<int64_t>({(int64_t)count, dev_cap, cap_of(k)});
        if (ncopy > 0) BMX_CUDA(cudaMemcpyAsync(pos_out[k], c->pos.p, (size_t)ncopy * 8, cudaMemcpyDeviceToHost, c->scan_stream));
        BMX_CUDA(cudaStreamSynchronize(c->scan_stream));   // c->pos is reused by the next pattern
        return BMX_OK;
    };
    // the text crosses PCIe once; then all patterns in one pass over the resident copy when the set is eligible
    // (bmx_multipat.cu), else pattern by pattern
    Ingest io;
    io.copy_only = true;
    int32_t m_min = ms[0];
    for (int32_t k = 1; k < npat; ++k) m_min = std::min(m_min, ms[k]);
    int rc = ingest_and_scan(*c, device, text, n, pats[0], m_min, 0, BMX_VARIANT_AUTO, &io);
    if (rc == BMX_E_NOMEM) {
        // larger than the device: every pattern streams the text through the ring on its own
        for (int32_t k = 0; k < npat; ++k) {
            Ingest one;
            one.want_cap = cap_of(k);
            if ((rc = ingest_and_scan(*c, device, text, n, pats[k], ms[k], 0, BMX_VARIANT_AUTO, &one)) != BMX_OK) return rc;
            counts[k] = one.count;
            if ((rc = fetch(k, one.count, one.dev_cap)) != BMX_OK) return rc;
        }
        return BMX_OK;
    }
    if (rc != BMX_OK) return rc;
    const unsigned char *d_text = static_cast<const unsigned char *>(c->text.p);
    if (multi_eligible(npat, ms)) {
        // device-side output buffers: a first guess per pattern (one hit per 64 bytes), grown to the counts if a
        // pattern turns out denser -- the resident text is simply scanned again
        std::vector<int64_t> dev_cap((size_t)npat, 0);
        for (int32_t k = 0; k < npat; ++k) dev_cap[(size_t)k] = first_pos_cap(n, ms[k], cap_of(k));
        for (int pass = 0; pass < 2; ++pass) {
            size_t total = 0;
            for (int32_t k = 0; k < npat; ++k) total += ((size_t)dev_cap[(size_t)k] * 8 + 255) & ~size_t(255);
            if ((rc = ensure_buf(*c, c->aux, std::max<size_t>(total, 256))) != BMX_OK) return rc;
            std::vector<int64_t *> outs((size_t)npat, nullptr);
            size_t at = 0;
            for (int32_t k = 0; k < npat; ++k) {
                if (dev_cap[(size_t)k] > 0) outs[(size_t)k] = reinterpret_cast<int64_t *>(static_cast<unsigned char *>(c->aux.p) + at);
                at += ((size_t)dev_cap[(size_t)k] * 8 + 255) & ~size_t(255);
            }
            if ((rc = multi_scan_resident(*c, d_text, n, npat, pats, ms, outs.data(), dev_cap.data(), counts, c->scan_stream)) != BMX_OK) return rc;
            bool grow = false;
            for (int32_t k = 0; k < npat; ++k) {
                const int64_t need = std::min<int64_t>(cap_of(k), (int64_t)counts[k]);
                if (need > dev_cap[(size_t)k]) {
                    dev_cap[(size_t)k] = need;
                    grow = true;
                }
            }
            if (!grow) {
                for (int32_t k = 0; k < npat; ++k) {
                    const int64_t ncopy = std::min<int64_t>({(int64_t)counts[k], dev_cap[(size_t)k], cap_of(k)});
                    if (ncopy > 0) BMX_CUDA(cudaMemcpyAsync(pos_out[k], outs[(size_t)k], (size_t)ncopy * 8, cudaMemcpyDeviceToHost, c->scan_stream));
                }
                BMX_CUDA(cudaStreamSynchronize(c->scan_stream));
                return BMX_OK;
            }
        }
        return fail(BMX_E_CUDA, "bmx_search_multi: position buffers did not converge");
    }
    for (int32_t k = 0; k < npat; ++k) {
        if (n < ms[k]) continue;
        uint64_t count = 0;
        int64_t dev_cap = 0;
        if ((rc = scan_resident(*c, d_text, n, pats[k], ms[k], BMX_VARIANT_AUTO, 0, cap_of(k), &count, &dev_cap, nullptr)) != BMX_OK) return rc;
        counts[k] = count;
        if ((rc = fetch(k, count, dev_cap)) != BMX_OK) return rc;
    }
    return BMX_OK;
}

int bmx_find_first(const char *text, int64_t n, const char *pat, int32_t m, int64_t *first_out)
{
    if (!first_out || !pat) return fail(BMX_E_BADARG, "bmx_find_first: pat/first_out must be non-NULL");
    if (int rc = check_text(text, n, "bmx_find_first")) return rc;
    if (int rc = check_pattern(m)) return rc;
    *first_out = -1;
    ThreadCtx *c = nullptr;
    if (int rc = current_ctx(&c)) return rc;
    if (n < m) return BMX_OK;
    if ((uint64_t)n > kFindMask) return fail(BMX_E_BADARG, "bmx_find_first: texts beyond 2^47 bytes are not supported");
    Ingest io;
    io.find_first = true;
    if (int rc = ingest_and_scan(*c, c->device, text, n, pat, m, 0, BMX_VARIANT_AUTO, &io)) return rc;
    *first_out = io.first;
    return BMX_OK;
}

int bmx_search_partitions(const char *text, const char *pat, const int32_t *se, int32_t *ans, const int32_t *gs,
                          const int32_t *bs, int32_t m, int32_t nparts)
{
    if (!pat || !se || !ans || nparts < 0 || (!text && nparts > 0))
        return fail(BMX_E_BADARG, "bmx_search_partitions: NULL argument or nparts < 0");
    if (int rc = check_pattern(m)) return rc;
    if (nparts == 0) return BMX_OK;

    // The reference hands its own tables to the kernel (BoyreMoore.cpp:268-269).  The device scan
    // keeps its own copy, so caller tables are only checked: a wrong table must not go unnoticed.
    if (gs || bs) {
        std::vector<int32_t> good((size_t)m);
        int32_t bad[256];
        build_bad_table(reinterpret_cast<const unsigned char *>(pat), m, bad);
        build_good_table(reinterpret_cast<const unsigned char *>(pat), m, good.data());
        if (gs)
            for (int32_t k = 1; k < m; ++k)
                if (gs[k] != good[(size_t)k]) return fail(BMX_E_TABLES, "gstable[%d] = %d, expected %d", k, gs[k], good[(size_t)k]);
        if (bs)
            for (int c = 0; c < 128; ++c)
                if (bs[c] != bad[c]) return fail(BMX_E_TABLES, "bstable[%d] = %d, expected %d", c, bs[c], bad[c]);
    }

    int64_t lo = INT64_MAX, hi = -1;
    for (int32_t id = 0; id < nparts; ++id) {
        if (se[2 * id] < 0) return fail(BMX_E_BADARG, "se[%d] = %d is negative", 2 * id, se[2 * id]);
        lo = std::min<int64_t>(lo, se[2 * id]);
        hi = std::max<int64_t>(hi, se[2 * id + 1]);
    }
    for (int32_t id = 0; id < nparts; ++id) ans[id] = 0;  // kernel1.cl:6
    const int64_t span = hi - lo + 1;
    if (span < m) return BMX_OK;

    ThreadCtx *c = nullptr;
    if (int rc = current_ctx(&c)) return rc;
    // One work-item of the reference = the occurrences lying fully inside its inclusive range (kernel1.cl:15,19):
    // range [s, e + 1) of the ranges search, which scans the covered bytes [lo, hi] once with positions and
    // answers every range from that one list (bmx_ranges.cu).  A range with e < s counts 0: it becomes empty.
    std::vector<int64_t> begin((size_t)nparts), end((size_t)nparts), offsets((size_t)nparts + 1);
    std::vector<uint64_t> counts((size_t)nparts, 0);
    for (int32_t id = 0; id < nparts; ++id) {
        const int64_t s = se[2 * id], e = (int64_t)se[2 * id + 1] + 1;
        begin[(size_t)id] = e < s ? lo : s;
        end[(size_t)id] = e < s ? lo : e;
    }
    if (int rc = search_ranges_host(*c, text, hi + 1, nparts, begin.data(), end.data(), lo, hi + 1, pat, m, nullptr, 0,
                                    counts.data(), offsets.data()))
        return rc;
    for (int32_t id = 0; id < nparts; ++id) ans[id] = (int32_t)counts[(size_t)id];
    return BMX_OK;
}

}  // extern "C"
