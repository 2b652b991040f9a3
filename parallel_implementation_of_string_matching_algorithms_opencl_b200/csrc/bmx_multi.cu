// bmx_multi.cu -- single-process multi-GPU entry points (bmx_mg_*): one host text cut into shards with (m-1)-byte
// halos and ingested over every GPU's own PCIe link (bmx_mg_search), or device-resident shards combined by the
// library's exchange step over NVLink peer memory (bmx_mg_search_device, bmx_exchange.cu).
//
// The reference has one device (BoyreMoore/BoyreMoore/BoyreMoore.cpp:217-219) and splits its text into word
// ranges WITHOUT overlap (:119-141), losing matches at the seams; here a shard owns the match START positions
// of its range and reads the halo behind it, so every occurrence is reported exactly once.
#include <cuda_runtime.h>

#include <algorithm>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "bmx_ctx.h"

using namespace bmx;

extern "C" {

struct bmx_mg {
    std::vector<int> devices;
    std::vector<ThreadCtx *> ctx;
    // device-resident flavour (bmx_mg_search_device): one exchange + one local position buffer per GPU
    std::vector<bmx_exchange *> xchg;
    std::vector<int64_t *> d_local_pos;
    int64_t xchg_tail_cap = -1;
};

namespace {

constexpr int64_t kMgHeadCap = 4096;

void mg_drop_exchange(bmx_mg *mg)
{
    for (size_t r = 0; r < mg->devices.size(); ++r) {
        cudaSetDevice(mg->devices[r]);
        if (r < mg->ctx.size() && mg->ctx[r]->scan_stream) cudaStreamSynchronize(mg->ctx[r]->scan_stream);
    }
    for (bmx_exchange *x : mg->xchg) bmx_exchange_destroy(x);
    mg->xchg.clear();
    for (size_t r = 0; r < mg->d_local_pos.size(); ++r) {
        cudaSetDevice(mg->devices[r]);
        if (mg->d_local_pos[r]) cudaFree(mg->d_local_pos[r]);
    }
    mg->d_local_pos.clear();
    mg->xchg_tail_cap = -1;
}

// Exchanges (and local position buffers of head + tail entries) able to ship lists of up to head + tail_cap positions.
int mg_ensure_exchange(bmx_mg *mg, int64_t tail_cap)
{
    if (!mg->xchg.empty() && mg->xchg_tail_cap >= tail_cap) return BMX_OK;
    mg_drop_exchange(mg);
    const int R = (int)mg->devices.size();
    int rc = BMX_OK;
    for (int r = 0; r < R && rc == BMX_OK; ++r) {
        bmx_exchange *x = nullptr;
        rc = bmx_exchange_create(mg->devices[(size_t)r], r, R, 0, kMgHeadCap, tail_cap, 4, &x);
        if (rc == BMX_OK) mg->xchg.push_back(x);
    }
    if (rc == BMX_OK) rc = bmx_exchange_connect_local(mg->xchg.data(), R);
    for (int r = 0; r < R && rc == BMX_OK; ++r) {
        int64_t *p = nullptr;
        cudaSetDevice(mg->devices[(size_t)r]);
        const cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&p), (size_t)(kMgHeadCap + tail_cap) * 8);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            rc = fail(e == cudaErrorMemoryAllocation ? BMX_E_NOMEM : BMX_E_CUDA, "bmx_mg_search_device: %s", cudaGetErrorString(e));
        } else {
            mg->d_local_pos.push_back(p);
        }
    }
    if (rc != BMX_OK) {
        const std::string keep_msg = bmx_last_error();
        mg_drop_exchange(mg);
        return fail(rc, "%s", keep_msg.c_str());
    }
    mg->xchg_tail_cap = tail_cap;
    return BMX_OK;
}

}  // namespace

int bmx_mg_create(int ngpus, bmx_mg **out)
{
    if (!out) return fail(BMX_E_BADARG, "bmx_mg_create: out is NULL");
    *out = nullptr;
    if (int rc = check_device(0)) return rc;
    int have = 0;
    BMX_CUDA(cudaGetDeviceCount(&have));
    if (ngpus <= 0) ngpus = have;
    if (ngpus > have) return fail(BMX_E_BADARG, "bmx_mg_create: %d GPUs requested, %d visible", ngpus, have);
    ScopedDevice keep;
    bmx_mg *mg = new (std::nothrow) bmx_mg();
    if (!mg) return fail(BMX_E_NOMEM, "out of host memory");
    for (int d = 0; d < ngpus; ++d) {
        ThreadCtx *c = new (std::nothrow) ThreadCtx();
        int rc = c ? BMX_OK : fail(BMX_E_NOMEM, "out of host memory");
        if (rc == BMX_OK) rc = bmx_scanner_create(d, &c->scanner);
        if (c) c->device = d;
        if (rc != BMX_OK) {
            delete c;
            bmx_mg_destroy(mg);
            return rc;
        }
        mg->devices.push_back(d);
        mg->ctx.push_back(c);
    }
    *out = mg;
    return BMX_OK;
}

void bmx_mg_destroy(bmx_mg *mg)
{
    if (!mg) return;
    ScopedDevice keep;
    mg_drop_exchange(mg);
    for (ThreadCtx *c : mg->ctx) delete c;   // ~ThreadCtx gives back the scanner, streams, events and buffers
    delete mg;
}

int bmx_mg_device_count(const bmx_mg *mg) { return mg ? (int)mg->devices.size() : 0; }

int bmx_mg_search(bmx_mg *mg, const char *text, int64_t n, const char *pat, int32_t m, int64_t *pos_out, int64_t pos_cap,
                  uint64_t *count_out, uint64_t *shard_counts)
{
    if (!mg || !count_out || !pat) return fail(BMX_E_BADARG, "bmx_mg_search: NULL argument");
    if (int rc = check_text(text, n, "bmx_mg_search")) return rc;
    if (pos_cap < 0) return fail(BMX_E_BADARG, "pos_cap < 0");
    if (int rc = check_pattern(m)) return rc;
    const int R = (int)mg->devices.size();
    *count_out = 0;
    for (int r = 0; r < R && shard_counts; ++r) shard_counts[r] = 0;
    if (n < m) return BMX_OK;

    // rank r owns the START positions [lo_r, hi_r) and reads (m-1) bytes of halo behind hi_r
    int64_t per = (n + R - 1) / R;
    per = (per + 15) & ~int64_t(15);
    struct Shard {
        int64_t lo = 0, hi = 0, end = 0, cap = 0, dev_cap = 0;
        int64_t *d_pos = nullptr;
        uint64_t count = 0;
        int rc = BMX_OK;
        std::string err;
    };
    std::vector<Shard> sh((size_t)R);
    std::vector<std::thread> workers;
    for (int r = 0; r < R; ++r) {
        Shard &s = sh[(size_t)r];
        s.lo = std::min<int64_t>(n, (int64_t)r * per);
        s.hi = std::min<int64_t>(n, s.lo + per);
        s.end = std::min<int64_t>(n, s.hi + m - 1);
        s.cap = pos_out ? std::min<int64_t>(pos_cap, s.hi - s.lo) : 0;
        if (s.end - s.lo < m) continue;
        workers.emplace_back([&, r]() {
            Shard &w = sh[(size_t)r];
            ThreadCtx &cx = *mg->ctx[(size_t)r];
            w.rc = ingest_shard(cx, mg->devices[(size_t)r], text + w.lo, w.end - w.lo, pat, m, w.lo, w.cap, &w.count, &w.dev_cap);
            w.d_pos = static_cast<int64_t *>(cx.pos.p);   // owned by the GPU's context
            if (w.rc != BMX_OK) w.err = bmx_last_error();
        });
    }
    for (auto &t : workers) t.join();

    int rc = BMX_OK;
    std::string err;
    uint64_t total = 0;
    for (int r = 0; r < R; ++r) {
        if (sh[(size_t)r].rc != BMX_OK && rc == BMX_OK) {
            rc = sh[(size_t)r].rc;
            err = sh[(size_t)r].err;
        }
        total += sh[(size_t)r].count;
        if (shard_counts) shard_counts[r] = sh[(size_t)r].count;
    }
    // gather: shard lists are ascending and shards are ordered, so concatenation is the sorted result
    ScopedDevice keep;
    int64_t off = 0;
    for (int r = 0; r < R; ++r) {
        Shard &s = sh[(size_t)r];
        cudaSetDevice(mg->devices[(size_t)r]);
        cudaStream_t st = mg->ctx[(size_t)r]->scan_stream;
        if (rc == BMX_OK && s.d_pos && s.cap > 0) {
            const int64_t have = std::min<int64_t>({(int64_t)s.count, s.cap, s.dev_cap});
            const int64_t ncopy = std::max<int64_t>(0, std::min<int64_t>(have, pos_cap - off));
            if (ncopy > 0 && cudaMemcpyAsync(pos_out + off, s.d_pos, (size_t)ncopy * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess) {
                rc = BMX_E_CUDA;
                err = "position gather failed";
            }
        }
        off += (int64_t)s.count;
    }
    for (int r = 0; r < R; ++r) {
        cudaSetDevice(mg->devices[(size_t)r]);
        if (mg->ctx[(size_t)r]->scan_stream && cudaStreamSynchronize(mg->ctx[(size_t)r]->scan_stream) != cudaSuccess && rc == BMX_OK) {
            rc = BMX_E_CUDA;
            err = "stream synchronisation failed";
        }
    }
    if (rc != BMX_OK) return fail(rc, "bmx_mg_search: %s", err.c_str());
    *count_out = total;
    return BMX_OK;
}


int bmx_mg_search_device(bmx_mg *mg, const void *const *d_text, const int64_t *n, const int64_t *pos_base, const char *pat,
                         int32_t m, int64_t *d_pos_out, int64_t pos_cap, uint64_t *count_out, uint64_t *shard_counts)
{
    if (!mg || !d_text || !n || !pos_base || !pat || !count_out) return fail(BMX_E_BADARG, "bmx_mg_search_device: NULL argument");
    if (pos_cap < 0) return fail(BMX_E_BADARG, "pos_cap < 0");
    if (int rc = check_pattern(m)) return rc;
    const int R = (int)mg->devices.size();
    for (int r = 0; r < R; ++r)
        if (n[r] < 0 || (!d_text[r] && n[r] > 0)) return fail(BMX_E_BADARG, "bmx_mg_search_device: bad shard %d (n=%lld)", r, (long long)n[r]);
    *count_out = 0;
    const bool want_pos = d_pos_out != nullptr && pos_cap > 0;
    ScopedDevice keep;
    int rc = BMX_OK;
    std::vector<uint64_t> counts((size_t)R, 0);
    uint64_t total = 0;
    int64_t tail_cap = std::max<int64_t>(mg->xchg_tail_cap, 0);
    for (int attempt = 0; attempt < 2 && rc == BMX_OK; ++attempt) {
        if ((rc = mg_ensure_exchange(mg, tail_cap)) != BMX_OK) break;
        const int64_t local_cap = want_pos ? kMgHeadCap + mg->xchg_tail_cap : 0;
        uint64_t seq = 0;
        for (int r = 0; r < R && rc == BMX_OK; ++r) {   // every launch is asynchronous: one host thread feeds all GPUs
            ThreadCtx *c = mg->ctx[(size_t)r];
            cudaSetDevice(mg->devices[(size_t)r]);
            if ((rc = ensure_streams(*c, 1)) != BMX_OK) break;
            if ((rc = bmx_scanner_set_pattern(c->scanner, pat, m, BMX_VARIANT_AUTO, c->scan_stream)) != BMX_OK) break;
            if ((rc = bmx_scanner_begin(c->scanner, want_pos ? mg->d_local_pos[(size_t)r] : nullptr, local_cap, c->scan_stream)) != BMX_OK) break;
            if ((rc = bmx_scanner_scan(c->scanner, d_text[r], n[r], pos_base[r], c->scan_stream)) != BMX_OK) break;
            rc = bmx_exchange_post(mg->xchg[(size_t)r], c->scanner, c->scan_stream, &seq);
        }
        for (int r = 0; r < R && rc == BMX_OK; ++r) {
            cudaSetDevice(mg->devices[(size_t)r]);
            rc = bmx_exchange_collect(mg->xchg[(size_t)r], r == 0 && want_pos ? d_pos_out : nullptr, pos_cap, mg->ctx[(size_t)r]->scan_stream, nullptr);
        }
        int64_t gathered = 0;
        for (int r = R - 1; r >= 0 && rc == BMX_OK; --r)
            rc = bmx_exchange_wait(mg->xchg[(size_t)r], seq, &total, counts.data(), &gathered);
        if (rc != BMX_OK) break;
        cudaSetDevice(mg->devices[0]);
        if (cudaStreamSynchronize(mg->ctx[0]->scan_stream) != cudaSuccess) {
            rc = fail(BMX_E_CUDA, "bmx_mg_search_device: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        if (!want_pos || gathered >= std::min<int64_t>((int64_t)total, pos_cap)) break;
        // a shard's list did not fit head + tail: size the transport for what the caller can still use and go again
        int64_t room = pos_cap, need = 0;
        for (int r = 0; r < R; ++r) {
            need = std::max<int64_t>(need, std::min<int64_t>((int64_t)counts[(size_t)r], room));
            room = std::max<int64_t>(0, room - (int64_t)counts[(size_t)r]);
        }
        if (need <= kMgHeadCap + mg->xchg_tail_cap) break;
        tail_cap = ((need - kMgHeadCap) + 4095) & ~int64_t(4095);
    }
    if (rc != BMX_OK) return rc;
    *count_out = total;
    for (int r = 0; r < R && shard_counts; ++r) shard_counts[r] = counts[(size_t)r];
    return BMX_OK;
}

}  // extern "C"
