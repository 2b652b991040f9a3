// bmx_abi.cu -- the C ABI of libbmx.so (include/bmx.h): host glue over the scan kernels.
//
// Replaces the reference's OpenCL host layer, BoyreMoore/BoyreMoore/BoyreMoore.cpp:192-313
// (context/queue :213-231, buffers :233-244, blocking writes :246-252, kernel + arguments
// :261-270, NDRange launch :273-280, blocking read of the counts :286, releases :299-312).
// There is no CPU fallback anywhere in this file: every scanning entry point needs a CUDA device.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "bmx_ctx.h"

namespace bmx {

// ---------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------
static thread_local char tl_error[512] = "";

int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(tl_error, sizeof tl_error, fmt, ap);
    va_end(ap);
    return code;
}

int check_device(int device)
{
    int n = 0;
    const cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        (void)cudaGetLastError();
        return fail(BMX_E_NODEVICE, "no CUDA device visible (%s); libbmx has no CPU path",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= n) return fail(BMX_E_BADARG, "device %d out of range (0..%d)", device, n - 1);
    return BMX_OK;
}

int check_text(const void *text, int64_t n, const char *who)
{
    if (n < 0 || (!text && n > 0)) return fail(BMX_E_BADARG, "%s: bad text (n=%lld)", who, (long long)n);
    return BMX_OK;
}

int check_pattern(int32_t m)
{
    if (m <= 0 || m > BMX_MAX_PATTERN)
        return fail(BMX_E_BADARG, "pattern length %d outside 1..%d (an empty pattern is rejected)", m, BMX_MAX_PATTERN);
    return BMX_OK;
}

int check_pattern_set(int32_t npat, const char *const *pats, const int32_t *ms, int64_t *const *outs, const int64_t *caps,
                      uint64_t *counts, const char *who)
{
    if (npat < 0 || (npat > 0 && (!pats || !ms || !counts))) return fail(BMX_E_BADARG, "%s: NULL argument or npat < 0", who);
    for (int32_t k = 0; k < npat; ++k) {
        if (!pats[k] || ms[k] <= 0 || ms[k] > BMX_MAX_PATTERN)
            return fail(BMX_E_BADARG, "pattern %d: length %d outside 1..%d or NULL (an empty pattern is rejected)", k, ms[k], BMX_MAX_PATTERN);
        if (outs && outs[k] && (!caps || caps[k] < 0)) return fail(BMX_E_BADARG, "pattern %d: pos_cap < 0 or missing", k);
        counts[k] = 0;
    }
    return BMX_OK;
}

}  // namespace bmx

using namespace bmx;

// ---------------------------------------------------------------------------------------------
// scanner (struct bmx_scanner: bmx_scanner.h)
// ---------------------------------------------------------------------------------------------
extern "C" {

int bmx_version(void) { return BMX_VERSION; }

const char *bmx_last_error(void) { return tl_error; }

int bmx_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return n;
}

int bmx_build_tables(const char *pat, int32_t m, int32_t bad[256], int32_t *good)
{
    if (!pat || m <= 0 || m > BMX_MAX_PATTERN || !bad || !good)
        return fail(BMX_E_BADARG, "bmx_build_tables: pat/bad/good must be non-NULL and 1 <= m <= %d", BMX_MAX_PATTERN);
    build_bad_table(reinterpret_cast<const unsigned char *>(pat), m, bad);
    build_good_table(reinterpret_cast<const unsigned char *>(pat), m, good);
    return BMX_OK;
}

int bmx_scanner_create(int device, bmx_scanner **out)
{
    if (!out) return fail(BMX_E_BADARG, "bmx_scanner_create: out is NULL");
    *out = nullptr;
    if (int rc = check_device(device)) return rc;
    BMX_CUDA(cudaSetDevice(device));
    bmx_scanner *s = new (std::nothrow) bmx_scanner();
    if (!s) return fail(BMX_E_NOMEM, "out of host memory");
    s->device = device;
    cudaError_t e = cudaMalloc(&s->d_ctrl, 64);
    if (e == cudaSuccess) e = cudaMemset(s->d_ctrl, 0, 64);
    if (e == cudaSuccess) e = cudaHostAlloc(&s->h_result, 64, cudaHostAllocMapped);
    if (e == cudaSuccess) {
        memset(s->h_result, 0, 64);
        e = cudaHostGetDevicePointer(reinterpret_cast<void **>(&s->d_result), s->h_result, 0);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_pat, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev_start);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev_stop);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev_k0);
    if (e == cudaSuccess) e = cudaEventCreate(&s->ev_k1);
    if (e != cudaSuccess) {
        bmx_scanner_destroy(s);
        return fail(e == cudaErrorMemoryAllocation ? BMX_E_NOMEM : BMX_E_CUDA, "bmx_scanner_create: %s",
                    cudaGetErrorString(e));
    }
    *out = s;
    return BMX_OK;
}

void bmx_scanner_destroy(bmx_scanner *s)
{
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->d_block) cudaFree(s->d_block);
    if (s->d_scratch) cudaFree(s->d_scratch);
    if (s->d_ctrl) cudaFree(s->d_ctrl);
    if (s->h_result) cudaFreeHost(s->h_result);
    if (s->ev_start) cudaEventDestroy(s->ev_start);
    if (s->ev_stop) cudaEventDestroy(s->ev_stop);
    if (s->ev_k0) cudaEventDestroy(s->ev_k0);
    if (s->ev_k1) cudaEventDestroy(s->ev_k1);
    if (s->ev_pat) cudaEventDestroy(s->ev_pat);
    (void)cudaGetLastError();
    delete s;
}

int bmx_scanner_set_pattern(bmx_scanner *s, const char *pat, int32_t m, int32_t variant, void *stream)
{
    if (!s || !pat) return fail(BMX_E_BADARG, "bmx_scanner_set_pattern: NULL argument");
    if (int rc = check_pattern(m)) return rc;
    const int32_t base = variant & ~BMX_IGNORE_CASE;
    if (base < BMX_VARIANT_AUTO || base > BMX_VARIANT_SHIFTAND)
        return fail(BMX_E_BADARG, "unknown variant %d", variant);
    BMX_CUDA(cudaSetDevice(s->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);

    const unsigned char *p = reinterpret_cast<const unsigned char *>(pat);
    // BMX_IGNORE_CASE: everything below works on the folded pattern.  A pattern without an ASCII letter is its own
    // fold and matches the same positions either way: it runs the exact kernels.
    std::vector<unsigned char> folded;
    bool fold = false;
    if (variant & BMX_IGNORE_CASE) {
        folded.resize((size_t)m);
        for (int32_t i = 0; i < m; ++i) {
            folded[(size_t)i] = ascii_lower(p[i]);
            fold = fold || (unsigned)((p[i] | 0x20u) - 'a') < 26u;   // an ASCII letter
        }
        p = folded.data();
    }
    const Filter filter = choose_filter(base, p, m);
    if (s->d_block && s->m == m && s->filter == filter && s->fold == fold && memcmp(s->pat.data(), p, (size_t)m) == 0) {
        // same pattern as last time (a caller searching many texts for one pattern): tables and device block stand.
        // The upload was ordered on pat_stream only; any other stream waits for it (an event wait, no copy).
        if (st != s->pat_stream) BMX_CUDA(cudaStreamWaitEvent(st, s->ev_pat, 0));
        return BMX_OK;
    }
    s->m = m;
    s->m_halo = 0;
    s->filter = filter;
    s->fold = fold;
    s->pat.assign(p, p + m);

    // Host image of the device block: tables once per pattern (BoyreMoore.cpp:153-190).
    const size_t good_off = 256 * sizeof(int32_t);
    const size_t pat_off = good_off + (size_t)m * sizeof(int32_t);
    const size_t bytes = ((pat_off + (size_t)m + 15) & ~size_t(15)) + 16;  // verification reads aligned word pairs
    std::vector<unsigned char> image(bytes, 0);
    build_bad_table(p, m, reinterpret_cast<int32_t *>(image.data()));
    build_good_table(p, m, reinterpret_cast<int32_t *>(image.data() + good_off));
    memcpy(image.data() + pat_off, p, (size_t)m);

    if (bytes > s->d_block_cap) {
        // the old block may still be read by scans in flight on `stream`
        BMX_CUDA(cudaStreamSynchronize(st));
        if (s->d_block) cudaFree(s->d_block);
        s->d_block = nullptr;
        s->d_block_cap = 0;
        BMX_CUDA(cudaMalloc(&s->d_block, bytes));
        s->d_block_cap = bytes;
    }
    // pageable source: the runtime stages it before returning, so `image` may die afterwards
    const cudaError_t up = cudaMemcpyAsync(s->d_block, image.data(), bytes, cudaMemcpyHostToDevice, st);
    if (up != cudaSuccess) {
        s->m = 0;   // nothing cached: the block holds no whole pattern
        return fail(BMX_E_CUDA, "pattern upload: %s", cudaGetErrorString(up));
    }
    BMX_CUDA(cudaEventRecord(s->ev_pat, st));
    s->pat_stream = st;

    s->proto = ScanArgs{};
    s->proto.m = m;
    s->proto.g_bad = reinterpret_cast<const int32_t *>(s->d_block);
    s->proto.g_good = reinterpret_cast<const int32_t *>(static_cast<unsigned char *>(s->d_block) + good_off);
    s->proto.g_pat = static_cast<const uint8_t *>(s->d_block) + pat_off;
    fill_filter_constants(filter, p, m, &s->proto);
    return BMX_OK;
}

int bmx_scanner_begin(bmx_scanner *s, int64_t *d_pos_out, int64_t pos_cap, void *stream)
{
    if (!s) return fail(BMX_E_BADARG, "bmx_scanner_begin: NULL scanner");
    if (pos_cap < 0) return fail(BMX_E_BADARG, "pos_cap < 0");
    BMX_CUDA(cudaSetDevice(s->device));
    s->d_pos_out = d_pos_out;
    s->pos_cap = d_pos_out ? pos_cap : 0;
    s->positions = d_pos_out != nullptr;
    s->scan_index = 0;
    s->find_epoch = 0;
    s->timing_open = false;
    s->stats = bmx_stats{};
    s->stats.variant = s->m > 0 ? filter_variant(s->filter) | (s->fold ? BMX_IGNORE_CASE : 0) : BMX_VARIANT_AUTO;
    // no device work here: the first scan of the search treats the carried state as zero (ScanArgs::first_scan)
    (void)stream;
    return BMX_OK;
}

int bmx_scanner_scan(bmx_scanner *s, const void *d_text, int64_t n, int64_t pos_base, void *stream)
{
    if (!s || s->m <= 0) return fail(BMX_E_BADARG, "bmx_scanner_scan: scanner has no pattern");
    if (int rc = check_text(d_text, n, "bmx_scanner_scan")) return rc;
    if (n < s->m) return BMX_OK;  // kernel1.cl:15,19: the loop is never entered
    BMX_CUDA(cudaSetDevice(s->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);

    ScanArgs a = s->proto;
    const uintptr_t addr = reinterpret_cast<uintptr_t>(d_text);
    const int64_t lead = (int64_t)(addr & 15u);
    a.vtext = reinterpret_cast<const uint8_t *>(addr - (uintptr_t)lead);
    a.vlen = lead + n;
    a.vmin = lead;
    a.vmax = lead + n - s->m;
    a.pos_bias = pos_base - lead;
    a.pos_out = s->d_pos_out;
    a.pos_cap = s->pos_cap;

    ScanLaunch launch{};
    if (int rc = plan_scan(s->device, s->filter, s->fold, s->m_halo ? s->m_halo : s->m, s->positions, &a, &launch)) return rc;

    // scratch: two "zero halves" [tickets 16 B | scan count u64 + pad | block_sum u32 x blocks | seg_count u16 x segs |
    //          item_flag u8 x items], each zero whenever a scan starts on it, followed by
    //          [block_base u64 x blocks | dense_list | mask16 u16 x chunks]                <- written before read.
    // Scans alternate between the halves: the expand kernel of scan i clears the half scan i-1 used, so in
    // steady state no memset sits between the kernels; a count-only scan resets its 32-byte header itself.
    const size_t off_bsum = 32;
    const size_t off_segc = off_bsum + (((size_t)a.num_blocks * 4 + 15) & ~size_t(15));
    // seg_count is padded to whole blocks: the expand kernel reads a block's 1024 counts with vector loads
    const size_t off_flag = off_segc + (size_t)a.num_blocks * kBlockSegs * 2;
    const size_t zero_bytes = s->positions ? off_flag + (((size_t)a.num_blocks * kExpandSplit + 15) & ~size_t(15)) : off_bsum;
    const size_t off_bbase = 0;
    const size_t off_dense = off_bbase + (((size_t)a.num_blocks * 8 + 15) & ~size_t(15));  // mask16 is read with 16-byte loads
    const size_t off_mask = off_dense + (((size_t)a.num_blocks * 4 + 15) & ~size_t(15));
    const size_t rest_bytes = s->positions ? off_mask + (size_t)a.num_segs * kSegChunks * 2 : 0;
    if (zero_bytes > s->zero_cap || 2 * s->zero_cap + rest_bytes > s->d_scratch_cap) {
        BMX_CUDA(cudaStreamSynchronize(st));
        if (s->d_scratch) cudaFree(s->d_scratch);
        s->d_scratch = nullptr;
        s->d_scratch_cap = 0;
        const size_t zcap = std::max<size_t>(s->zero_cap, ((zero_bytes + zero_bytes / 8 + 255) & ~size_t(255)));
        const size_t want = std::max<size_t>(2 * zcap + rest_bytes + rest_bytes / 8, 1 << 20);
        BMX_CUDA(cudaMalloc(&s->d_scratch, want));
        s->d_scratch_cap = want;
        s->zero_cap = zcap;
        BMX_CUDA(cudaMemsetAsync(s->d_scratch, 0, 2 * zcap, st));
        s->dirty[0] = s->dirty[1] = 0;
        s->cur_half = 0;
    }
    const int half = s->cur_half;
    unsigned char *base = static_cast<unsigned char *>(s->d_scratch) + (size_t)half * s->zero_cap;
    unsigned char *rest = static_cast<unsigned char *>(s->d_scratch) + 2 * s->zero_cap;
    if (s->dirty[half]) {  // not reached by alternating scans; keeps any other call order correct
        BMX_CUDA(cudaMemsetAsync(base, 0, s->dirty[half], st));
        s->dirty[half] = 0;
    }
    a.tile_counter = reinterpret_cast<uint32_t *>(base);
    a.scan_count = reinterpret_cast<unsigned long long *>(base + 16);
    a.block_sum = reinterpret_cast<uint32_t *>(base + off_bsum);
    a.seg_count = reinterpret_cast<uint16_t *>(base + off_segc);
    a.item_flag = base + off_flag;
    a.block_base = reinterpret_cast<unsigned long long *>(rest + off_bbase);
    a.dense_list = reinterpret_cast<uint32_t *>(rest + off_dense);
    a.mask16 = reinterpret_cast<uint16_t *>(rest + off_mask);
    a.zero_ptr = static_cast<unsigned char *>(s->d_scratch) + (size_t)(1 - half) * s->zero_cap;
    a.zero_vec16 = s->positions ? (uint32_t)((s->dirty[1 - half] + 15) / 16) : 0u;
    a.carry_in = s->d_ctrl + (s->scan_index & 1u);
    a.carry_out = s->d_ctrl + ((s->scan_index + 1u) & 1u);
    a.count_acc = s->d_ctrl + 2;
    a.first_scan = s->scan_index == 0 ? 1u : 0u;
    a.host_count = s->d_result;
    a.first_key = s->d_ctrl + 4;
    a.find_epoch = s->positions ? 0u : s->find_epoch;

    if (s->timing_level >= 1 && !s->timing_open) {
        BMX_CUDA(cudaEventRecord(s->ev_start, st));
        s->timing_open = true;
    }
    if (s->timing_level >= 2) BMX_CUDA(cudaEventRecord(s->ev_k0, st));
    if (int rc = launch_scan(a, launch, s->positions, st)) return rc;
    if (s->timing_level >= 2) BMX_CUDA(cudaEventRecord(s->ev_k1, st));
    if (s->positions) {
        s->dirty[half] = zero_bytes;
        if (int rc = launch_emit(a, st)) return rc;
        s->dirty[1 - half] = 0;   // cleared by the expand kernel just enqueued
        s->cur_half = 1 - half;
    }
    if (s->timing_level >= 1) BMX_CUDA(cudaEventRecord(s->ev_stop, st));

    s->scan_index += 1;
    s->stats.kernel_launches += s->positions ? 2 : 1;
    s->stats.grid = launch.grid;
    s->stats.stages = (int32_t)a.stages;
    s->stats.tile_bytes = launch.tile_bytes;
    s->stats.smem_bytes = (int32_t)launch.smem_bytes;
    s->stats.tiles += a.num_tiles;
    return BMX_OK;
}

int bmx_scanner_set_timing(bmx_scanner *s, int level)
{
    if (!s || level < 0 || level > 2) return fail(BMX_E_BADARG, "bmx_scanner_set_timing: level must be 0, 1 or 2");
    s->timing_level = level;
    return BMX_OK;
}

int bmx_scanner_export_result(bmx_scanner *s, void *d_dst, int64_t head, void *stream)
{
    if (!s || !d_dst || head < 0) return fail(BMX_E_BADARG, "bmx_scanner_export_result: bad argument");
    BMX_CUDA(cudaSetDevice(s->device));
    const unsigned long long *src = result_slot(s);
    return launch_export_result(src, s->d_pos_out, s->pos_cap, d_dst, s->positions ? head : 0, stream);
}

int bmx_scanner_finish(bmx_scanner *s, uint64_t *count_out, bmx_stats *stats, void *stream)
{
    if (!s || !count_out) return fail(BMX_E_BADARG, "bmx_scanner_finish: NULL argument");
    BMX_CUDA(cudaSetDevice(s->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // the last CTA of every scan stores the running count into host-mapped memory: no copy, one synchronisation
    BMX_CUDA(cudaStreamSynchronize(st));
    *count_out = s->scan_index ? (uint64_t)*static_cast<volatile unsigned long long *>(s->h_result) : 0;
    if (s->timing_open) {
        float ms = 0.f;
        BMX_CUDA(cudaEventElapsedTime(&ms, s->ev_start, s->ev_stop));
        s->stats.device_ms = ms;
        if (s->timing_level >= 2 && s->stats.kernel_launches > 0 && cudaEventElapsedTime(&ms, s->ev_k0, s->ev_k1) == cudaSuccess)
            s->stats.scan_kernel_ms = ms;
    }
    if (stats) *stats = s->stats;
    return BMX_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// one cached scanner + streams + buffers per (host thread, device) for the convenience entry points (bmx_ctx.h)
// ---------------------------------------------------------------------------------------------
namespace bmx {

void ThreadCtx::release_buffers()
{
    if (device < 0) return;
    {
        ScopedDevice keep;
        if (cudaSetDevice(device) == cudaSuccess) {
            if (copy_stream) cudaStreamSynchronize(copy_stream);
            if (scan_stream) cudaStreamSynchronize(scan_stream);
            for (DevBuf *b : {&text, &pos, &misc, &aux}) {
                if (b->p) cudaFree(b->p);
                *b = DevBuf{};
            }
            for (int i = 0; i < kBounce; ++i) {
                if (bounce[i]) cudaFreeHost(bounce[i]);
                bounce[i] = nullptr;
            }
            bounce_bytes = 0;
            if (h_small) cudaFreeHost(h_small);
            h_small = nullptr;
        }
    }
    (void)cudaGetLastError();
}

ThreadCtx::~ThreadCtx()
{
    if (device < 0) return;
    // at process exit the CUDA runtime may already be gone: every call below then fails harmlessly
    release_buffers();
    {
        ScopedDevice keep;
        if (cudaSetDevice(device) == cudaSuccess) {
            if (scanner) bmx_scanner_destroy(scanner);
            if (copy_stream) cudaStreamDestroy(copy_stream);
            if (scan_stream) cudaStreamDestroy(scan_stream);
            for (cudaEvent_t e : events) cudaEventDestroy(e);
        }
        scanner = nullptr;
    }
    (void)cudaGetLastError();
}

static thread_local ThreadCtx tl_ctx[kMaxDevices];

int get_ctx(int device, ThreadCtx **out)
{
    if (int rc = check_device(device)) return rc;
    if (device >= kMaxDevices) return fail(BMX_E_BADARG, "device index %d too large", device);
    ThreadCtx &c = tl_ctx[device];
    BMX_CUDA(cudaSetDevice(device));
    if (!c.scanner) {
        if (int rc = bmx_scanner_create(device, &c.scanner)) return rc;
        c.device = device;
    }
    *out = &c;
    return BMX_OK;
}

int current_ctx(ThreadCtx **out)
{
    int device = 0;
    if (int rc = check_device(0)) return rc;
    BMX_CUDA(cudaGetDevice(&device));
    return get_ctx(device, out);
}

int ensure_streams(ThreadCtx &c, size_t nevents)
{
    if (!c.copy_stream) BMX_CUDA(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
    if (!c.scan_stream) BMX_CUDA(cudaStreamCreateWithFlags(&c.scan_stream, cudaStreamNonBlocking));
    while (c.events.size() < nevents) {
        cudaEvent_t e;
        BMX_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        c.events.push_back(e);
    }
    return BMX_OK;
}

int ensure_buf(ThreadCtx &c, DevBuf &b, size_t bytes)
{
    if (bytes <= b.cap) return BMX_OK;
    if (b.p) {
        if (c.copy_stream) BMX_CUDA(cudaStreamSynchronize(c.copy_stream));
        if (c.scan_stream) BMX_CUDA(cudaStreamSynchronize(c.scan_stream));
        cudaFree(b.p);
        b = DevBuf{};
    }
    const size_t want = (bytes + (size_t(1) << 20) - 1) & ~((size_t(1) << 20) - 1);
    BMX_CUDA(cudaMalloc(&b.p, want));
    b.cap = want;
    return BMX_OK;
}

// Starts a find-first search on s: count-only kernels that also keep the smallest hit in d_ctrl[4] and stop early.
int scanner_begin_find(bmx_scanner *s, void *stream)
{
    if (int rc = bmx_scanner_begin(s, nullptr, 0, stream)) return rc;
    if (s->find_epochs_used >= 65000u) {   // 16 bits of epoch: clear the key word before they wrap
        BMX_CUDA(cudaMemsetAsync(s->d_ctrl + 4, 0, sizeof(unsigned long long), static_cast<cudaStream_t>(stream)));
        s->find_epochs_used = 0;
    }
    s->find_epoch = ++s->find_epochs_used;
    return BMX_OK;
}

int search_once(bmx_scanner *s, const char *pat, int32_t m, int32_t variant, const void *d_text, int64_t n, int64_t pos_base,
                int64_t *d_pos, int64_t pos_cap, uint64_t *count, bmx_stats *stats, void *stream)
{
    int rc = bmx_scanner_set_pattern(s, pat, m, variant, stream);
    if (rc == BMX_OK) rc = bmx_scanner_begin(s, d_pos, pos_cap, stream);
    if (rc == BMX_OK) rc = bmx_scanner_scan(s, d_text, n, pos_base, stream);
    if (rc == BMX_OK) rc = bmx_scanner_finish(s, count, stats, stream);
    return rc;
}

}  // namespace bmx

extern "C" {

int bmx_release_memory(int device)
{
    for (int d = 0; d < kMaxDevices; ++d)
        if (device < 0 || d == device) tl_ctx[d].release_buffers();
    return BMX_OK;
}

int bmx_search_device_ex(const void *d_text, int64_t n, const char *pat, int32_t m, int64_t pos_base,
                         int64_t *d_pos_out, int64_t pos_cap, uint64_t *count_out, int32_t variant,
                         bmx_stats *stats, void *stream)
{
    if (!count_out || !pat) return fail(BMX_E_BADARG, "bmx_search_device: pat/count_out must be non-NULL");
    if (int rc = check_text(d_text, n, "bmx_search_device")) return rc;
    if (pos_cap < 0) return fail(BMX_E_BADARG, "pos_cap < 0");
    ThreadCtx *c = nullptr;
    if (int rc = current_ctx(&c)) return rc;
    // CUDA events between the kernels cost microseconds per call: only a caller that asks for the times pays
    ScopedTiming timing(c->scanner, stats ? 2 : 0);
    return search_once(c->scanner, pat, m, variant, d_text, n, pos_base, d_pos_out, pos_cap, count_out, stats, stream);
}

int bmx_search_device(const void *d_text, int64_t n, const char *pat, int32_t m, int64_t *d_pos_out,
                      int64_t pos_cap, uint64_t *count_out, float *device_ms, void *stream)
{
    bmx_stats st{};
    const int rc = bmx_search_device_ex(d_text, n, pat, m, 0, d_pos_out, pos_cap, count_out, BMX_VARIANT_AUTO,
                                        device_ms ? &st : nullptr, stream);
    if (rc == BMX_OK && device_ms) *device_ms = st.device_ms;
    return rc;
}

// First occurrence with a device-side stop.  ONE count-only scan over the whole text: every warp that finds a
// match folds its smallest start into a key word (atomicMax of epoch | ~position), the producer warps read that
// word before every tile fetch and stop fetching tiles that begin behind the best match (tiles are handed out
// in text order, so everything in front of it is already in flight), and the CTA that finishes last stores the
// result into host-mapped memory.  A miss costs one plain scan; an early match costs the launch plus the tiles
// in flight -- the in-kernel break of the vendored sample (boyer-moore.cu:62-86) without its race.
int bmx_find_first_device(const void *d_text, int64_t n, const char *pat, int32_t m, int64_t *first_out, void *stream)
{
    if (!first_out || !pat) return fail(BMX_E_BADARG, "bmx_find_first_device: pat/first_out must be non-NULL");
    if (int rc = check_text(d_text, n, "bmx_find_first_device")) return rc;
    *first_out = -1;
    ThreadCtx *c = nullptr;
    if (int rc = current_ctx(&c)) return rc;
    bmx_scanner *s = c->scanner;
    if (int rc = bmx_scanner_set_pattern(s, pat, m, BMX_VARIANT_AUTO, stream)) return rc;
    if (n < m) return BMX_OK;
    if ((uint64_t)n > kFindMask) return fail(BMX_E_BADARG, "bmx_find_first_device: texts beyond 2^47 bytes are not supported");
    ScopedTiming timing(s, 0);
    int rc = scanner_begin_find(s, stream);
    if (rc == BMX_OK) rc = bmx_scanner_scan(s, d_text, n, 0, stream);
    uint64_t partial = 0;
    if (rc == BMX_OK) rc = bmx_scanner_finish(s, &partial, nullptr, stream);
    if (rc == BMX_OK) *first_out = (int64_t) static_cast<volatile unsigned long long *>(s->h_result)[1];
    return rc;
}

int bmx_synth_fill_device(void *d_text, int64_t offset, int64_t len, uint64_t seed, const unsigned char *alphabet,
                          int32_t sigma, void *stream)
{
    if (len < 0 || offset < 0 || (!d_text && len > 0) || !alphabet || sigma < 1 || sigma > 256)
        return fail(BMX_E_BADARG, "bmx_synth_fill_device: bad argument");
    if (int rc = check_device(0)) return rc;
    return launch_synth_fill(d_text, offset, len, seed, alphabet, sigma, stream);
}

}  // extern "C"
