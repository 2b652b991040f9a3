// bmx_dict.cu -- dictionary search (grep -F -f wordlist): up to 65536 patterns in ONE pass over the text, the matches
// reported in text order as (position, pattern) pairs.  DESIGN §3.11.
//
//   create   the candidate table of bmx_search_multi (bmx_multipat.cu: fill_set_tables), built ONCE per dictionary
//            into a device block the handle owns, with its geometry set by K: an exact table of the next power of two
//            >= 8K slots (4 residues per pattern, load <= 1/2), a directory and a blob of K patterns, and a "home
//            slot occupied" bit array folded to at most 2^kDictMaxOccLog2 bits.  Block layout:
//            [bitmap 32 KiB | occupancy bits | table | directory | blob], the first two or three staged as they lie.
//   scan     the scan kernel's kDict instance: the same bitmap probe per aligned text word as kMulti; a flagged word
//            asks the staged occupancy bits (one shared-memory load) before it walks the table, which is staged into
//            shared memory up to 2^kDictMaxSmemSlotsLog2 slots and read from global memory (L2) above that.  Exact
//            per-pattern counters (sized K, per-call scratch) and the UNION hit mask -> the ordinary ordered
//            emission -> U, the ascending list of starts at which any pattern matches (the context's position buffer).
//   pairs    for each u in U in parallel: the residue r = (-u) mod 4 in V space, the aligned gram at u + r hashed
//            exactly as the scan hashes it, the table entries with that hash and residue compared with the text:
//            c(u) >= 1 matching patterns.  Every pattern has m >= m_min >= q + 3, so its residue-r gram is in the
//            table and the walk finds every pattern that matches at u.  dict_count_kernel writes c(u) and the
//            smallest k, per-CTA sums and (last CTA) the CTA bases; dict_write_kernel ranks every u by a block scan
//            and writes its pairs, k ascending, where the rank is below cap.
// U needs at most cap entries for the first cap pairs (c(u) >= 1); a text denser than the first guess is scanned
// again with room for them (the grow-and-rerun rule of multi_scan_resident).
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cstring>
#include <vector>

#include "bmx_ctx.h"

using namespace bmx;

struct bmx_dict {
    int device = 0;
    int32_t npat = 0;
    SetHash sh;
    uint32_t slots_log2 = 0, occ_log2 = 0, table_smem = 0;
    unsigned char *d_image = nullptr;
    size_t off_table = 0, off_dir = 0, off_blob = 0, blob_bytes = 0;
};

namespace {

constexpr int kPairThreads = 256;
constexpr int kPairBatch = 8;   // pattern ids a thread collects per table walk when several patterns match at one start

struct DictCtrl {               // zeroed per call; copied to the host behind the kernels
    unsigned long long total;   // pairs the held part of U yields
    unsigned int ticket;        // dict_count_kernel CTAs done
    unsigned int pad;
};

struct PairArgs {
    const int64_t *U;
    const unsigned long long *ucount;   // |U| (the scan's count, on the device)
    int64_t ucap;                       // entries of U the scan could write
    const uint8_t *text;
    int64_t n;
    uint32_t lead;                      // d_text & 15: V-space offset of text[0]
    SetHash sh;
    const uint2 *table, *dir;
    const uint8_t *blob;
    uint32_t slots_log2;
};

// The entries of U this CTA owns: a contiguous span, the grid covering the held part of U whatever its length.
__device__ __forceinline__ void cta_span(const PairArgs &P, int64_t *lo, int64_t *hi)
{
    const int64_t H = min((int64_t)*P.ucount, P.ucap), per = (H + gridDim.x - 1) / gridDim.x;
    *lo = min(H, (int64_t)blockIdx.x * per);
    *hi = min(H, *lo + per);
}

// Calls f(k) for every pattern k that matches at text start u, in table order.
template <typename F>
__device__ __forceinline__ void for_each_match(const PairArgs &P, int64_t u, F f)
{
    const uint32_t r = (uint32_t)(-(u + (int64_t)P.lead)) & 3u;   // pattern byte r lies on a word boundary of V
    if (u + r + 4 + P.sh.q2 + P.sh.q3 > P.n) return;              // (never for a start in U: m >= q + 3)
    const uint32_t h = set_gram_hash(P.sh, P.text + u + r);
    const uint32_t mask = (1u << P.slots_log2) - 1u;
    for (uint32_t slot = (h * kMultiSlotMul) >> (32 - P.slots_log2);; slot = (slot + 1) & mask) {
        const uint2 e = __ldg(P.table + slot);
        if (e.y == 0u) break;
        if (e.x != h || (e.y & 3u) != r) continue;
        const int32_t k = (int32_t)((e.y >> 2) & 0xFFFFu);
        const uint2 d = __ldg(P.dir + k);
        const int32_t mk = (int32_t)d.y;
        if (u + mk > P.n) continue;
        const uint8_t *pk = P.blob + d.x, *t = P.text + u;
        bool same = true;
        for (int32_t i = 0; same && i < mk; ++i) same = __ldg(t + i) == __ldg(pk + i);
        if (same) f(k);
    }
}

__global__ void __launch_bounds__(kPairThreads) dict_count_kernel(const PairArgs P, uint2 *cinfo, unsigned long long *cta_sum, DictCtrl *ctrl)
{
    int64_t lo, hi;
    cta_span(P, &lo, &hi);
    unsigned long long sum = 0;
    for (int64_t i = lo + threadIdx.x; i < hi; i += kPairThreads) {
        uint32_t c = 0, kmin = 0xFFFFFFFFu;
        for_each_match(P, P.U[i], [&](int32_t k) {
            ++c;
            kmin = min(kmin, (uint32_t)k);
        });
        cinfo[i] = make_uint2(c, kmin);
        sum += c;
    }
    unsigned long long cta_total = 0;
    (void)cta_exclusive_scan<kPairThreads>(sum, &cta_total);
    __shared__ bool last;
    if (threadIdx.x == 0) {
        cta_sum[blockIdx.x] = cta_total;
        __threadfence();
        last = atomicAdd(&ctrl->ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    // the last CTA: per-CTA sums -> exclusive bases, in place (range_rank_kernel's idiom, DESIGN §3.9)
    const int64_t G = gridDim.x, per = (G + kPairThreads - 1) / kPairThreads;
    const int64_t glo = min(G, (int64_t)threadIdx.x * per), ghi = min(G, glo + per);
    unsigned long long local = 0;
    for (int64_t g = glo; g < ghi; ++g) local += __ldcg(cta_sum + g);
    unsigned long long total = 0;
    unsigned long long run = cta_exclusive_scan<kPairThreads>(local, &total);
    for (int64_t g = glo; g < ghi; ++g) {
        const unsigned long long v = __ldcg(cta_sum + g);
        cta_sum[g] = run;
        run += v;
    }
    if (threadIdx.x == 0) ctrl->total = total;
}

__global__ void __launch_bounds__(kPairThreads) dict_write_kernel(const PairArgs P, const uint2 *cinfo, const unsigned long long *cta_base,
                                                                  int64_t pos_base, int64_t *pos_out, int32_t *pat_out, int64_t cap)
{
    int64_t lo, hi;
    cta_span(P, &lo, &hi);
    unsigned long long run = cta_base[blockIdx.x];
    for (int64_t b = lo; b < hi && (int64_t)run < cap; b += kPairThreads) {   // (both bounds are the same for the whole CTA)
        const int64_t i = b + threadIdx.x;
        const uint2 ci = i < hi ? cinfo[i] : make_uint2(0u, 0u);
        unsigned long long step = 0;
        const int64_t rank = (int64_t)(run + cta_exclusive_scan<kPairThreads>(ci.x, &step));
        run += step;
        if (ci.x == 0 || rank >= cap) continue;
        const int64_t u = P.U[i];
        if (ci.x == 1) {   // the common case: the count pass already named the pattern
            pos_out[rank] = u + pos_base;
            pat_out[rank] = (int32_t)ci.y;
            continue;
        }
        // several patterns at u (shared prefixes, duplicates): k ascending, up to kPairBatch ids per table walk
        const int64_t end = min(cap, rank + (int64_t)ci.x);
        int64_t at = rank;
        int32_t last = -1;
        while (at < end) {
            int32_t best[kPairBatch];   // the smallest ids above `last`, ascending (compare-and-swap insertion, in registers)
#pragma unroll
            for (int j = 0; j < kPairBatch; ++j) best[j] = INT32_MAX;
            for_each_match(P, u, [&](int32_t k) {
                if (k <= last) return;
#pragma unroll
                for (int j = 0; j < kPairBatch; ++j) {
                    if (k < best[j]) {
                        const int32_t t = best[j];
                        best[j] = k;
                        k = t;
                    }
                }
            });
            if (best[0] == INT32_MAX) break;   // (never: the count pass found ci.x patterns here)
#pragma unroll
            for (int j = 0; j < kPairBatch; ++j) {
                if (best[j] != INT32_MAX && at < end) {
                    pos_out[at] = u + pos_base;
                    pat_out[at] = best[j];
                    last = best[j];
                    ++at;
                }
            }
        }
    }
}

int sm_count(int device)
{
    int sms = 148;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) {
        (void)cudaGetLastError();
        sms = 148;
    }
    return sms;
}

}  // namespace

namespace bmx {

// All patterns of d over device-resident text d_text[0..n): exact counts (host), and the first cap pairs into the
// device arrays d_pos / d_pat (cap == 0: counts only).  Synchronous on st.
int dict_search_resident(ThreadCtx &c, const bmx_dict *d, const unsigned char *d_text, int64_t n, int64_t pos_base, int64_t *d_pos,
                         int32_t *d_pat, int64_t cap, uint64_t *counts, uint64_t *total_out, cudaStream_t st)
{
    const int32_t K = d->npat, m_min = d->sh.m_min;
    std::fill(counts, counts + K, 0ull);
    *total_out = 0;
    if (n < m_min) return BMX_OK;
    int64_t cap_u = cap > 0 ? first_pos_room(c, n, m_min, std::min<int64_t>(cap, n - m_min + 1)) : 0;

    bmx_scanner *s = c.scanner;
    // the scanner leaves single-pattern mode: its cached pattern block no longer describes proto
    s->filter = kDict;
    s->fold = false;
    s->pat.clear();
    s->proto = ScanArgs{};
    s->proto.m = m_min;
    s->proto.hmul = d->sh.hmul;
    s->proto.hmul2 = d->sh.hmul2;
    s->proto.g_mbits = reinterpret_cast<const uint32_t *>(d->d_image);
    s->proto.g_mtable = reinterpret_cast<const uint2 *>(d->d_image + d->off_table);
    s->proto.g_mdir = reinterpret_cast<const uint2 *>(d->d_image + d->off_dir);
    s->proto.g_mblob = d->d_image + d->off_blob;
    s->proto.npat = (uint32_t)K;
    s->proto.multi_blob_smem = d->blob_bytes <= (size_t)kPatSmemMax * 4 ? (uint32_t)d->blob_bytes : 0u;   // SmemCtl::good holds kPatSmemMax ints
    s->proto.mslots_log2 = d->slots_log2;
    s->proto.mtable_smem = d->table_smem;
    s->proto.mocc_log2 = d->occ_log2;
    s->m = m_min;
    s->m_halo = d->sh.m_max;
    ScopedTiming timing(s, 0);

    PairArgs P{};
    P.text = d_text;
    P.n = n;
    P.lead = (uint32_t)(reinterpret_cast<uintptr_t>(d_text) & 15u);
    P.sh = d->sh;
    P.table = s->proto.g_mtable;
    P.dir = s->proto.g_mdir;
    P.blob = s->proto.g_mblob;
    P.slots_log2 = d->slots_log2;

    // scratch: [DictCtrl | counters K | CTA sums G | (c, smallest k) per entry of U]; from here on every failure breaks
    // out of the loop, so that the scanner leaves dictionary mode below
    const size_t off_counts = 256, off_sum = off_counts + (((size_t)K * 8 + 255) & ~size_t(255));
    std::vector<unsigned long long> h_counts((size_t)K, 0);
    DictCtrl h_ctrl{};
    int rc = BMX_OK;
    for (int pass = 0; pass < 2 && rc == BMX_OK; ++pass) {
        const int64_t G = std::max<int64_t>(1, std::min<int64_t>((cap_u + kPairThreads - 1) / kPairThreads, (int64_t)sm_count(c.device) * 4));
        const size_t off_info = off_sum + (((size_t)G * 8 + 255) & ~size_t(255));
        if (cap_u > 0 && (rc = ensure_buf(c, c.pos, (size_t)cap_u * 8)) != BMX_OK) break;
        if ((rc = ensure_buf(c, c.misc, off_info + (size_t)cap_u * 8)) != BMX_OK) break;
        unsigned char *scratch = static_cast<unsigned char *>(c.misc.p);
        DictCtrl *ctrl = reinterpret_cast<DictCtrl *>(scratch);
        unsigned long long *d_counts = reinterpret_cast<unsigned long long *>(scratch + off_counts);
        if (cudaMemsetAsync(scratch, 0, off_counts + (size_t)K * 8, st) != cudaSuccess) {
            rc = fail(BMX_E_CUDA, "bmx_dict_search: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        s->proto.mcounts = d_counts;
        int64_t *U = cap_u > 0 ? static_cast<int64_t *>(c.pos.p) : nullptr;
        if ((rc = bmx_scanner_begin(s, U, cap_u, st)) != BMX_OK) break;
        if ((rc = bmx_scanner_scan(s, d_text, n, 0, st)) != BMX_OK) break;
        if (U) {
            P.U = U;
            P.ucount = result_slot(s);
            P.ucap = cap_u;
            uint2 *cinfo = reinterpret_cast<uint2 *>(scratch + off_info);
            unsigned long long *cta_sum = reinterpret_cast<unsigned long long *>(scratch + off_sum);
            dict_count_kernel<<<(unsigned)G, kPairThreads, 0, st>>>(P, cinfo, cta_sum, ctrl);
            dict_write_kernel<<<(unsigned)G, kPairThreads, 0, st>>>(P, cinfo, cta_sum, pos_base, d_pos, d_pat, cap);
            if (cudaError_t e = cudaGetLastError(); e != cudaSuccess) {
                rc = fail(BMX_E_CUDA, "dictionary pair kernels: %s", cudaGetErrorString(e));
                break;
            }
        }
        if (cudaMemcpyAsync(h_counts.data(), d_counts, (size_t)K * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaMemcpyAsync(&h_ctrl, ctrl, sizeof h_ctrl, cudaMemcpyDeviceToHost, st) != cudaSuccess) {
            rc = fail(BMX_E_CUDA, "bmx_dict_search: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        uint64_t ucount = 0;
        if ((rc = bmx_scanner_finish(s, &ucount, nullptr, st)) != BMX_OK) break;   // synchronises st
        uint64_t total = 0;
        for (int32_t k = 0; k < K; ++k) total += h_counts[(size_t)k];
        *total_out = total;
        if (!U) break;
        if ((int64_t)ucount <= cap_u && h_ctrl.total != total) {   // U is whole: its pairs are all the pairs
            rc = fail(BMX_E_CUDA, "bmx_dict_search: %llu pairs from the start list, %llu counted", (unsigned long long)h_ctrl.total,
                      (unsigned long long)total);
            break;
        }
        if ((int64_t)h_ctrl.total >= std::min<int64_t>((int64_t)total, cap) || (int64_t)ucount <= cap_u) break;
        cap_u = std::min<int64_t>((int64_t)ucount, cap);   // U was cut short before the first cap pairs: room for them
    }
    s->m_halo = 0;
    s->m = 0;   // the scanner has no single pattern until the next set_pattern
    if (rc != BMX_OK) return rc;
    for (int32_t k = 0; k < K; ++k) counts[k] = h_counts[(size_t)k];
    return BMX_OK;
}

}  // namespace bmx

namespace {

int check_search(const bmx_dict *d, const void *text, int64_t n, const void *pos_out, const void *pat_out, int64_t cap,
                 const uint64_t *counts, const uint64_t *total_out, const char *who)
{
    if (!d || !counts || !total_out) return fail(BMX_E_BADARG, "%s: NULL dictionary, counts or total_out", who);
    if (int rc = check_text(text, n, who)) return rc;
    if (cap < 0) return fail(BMX_E_BADARG, "%s: cap < 0", who);
    if ((pos_out == nullptr) != (pat_out == nullptr))
        return fail(BMX_E_BADARG, "%s: position and pattern outputs must both be given or both be NULL", who);
    return BMX_OK;
}

}  // namespace

extern "C" {

int bmx_dict_create(int device, int32_t npat, const char *const *pats, const int32_t *ms, bmx_dict **out)
{
    if (!out) return fail(BMX_E_BADARG, "bmx_dict_create: NULL out");
    *out = nullptr;
    if (npat < 1 || npat > kDictMaxPatterns || !pats || !ms)
        return fail(BMX_E_BADARG, "bmx_dict_create: need 1 <= npat <= %d patterns (got %d) and non-NULL pats / ms", kDictMaxPatterns, npat);
    for (int32_t k = 0; k < npat; ++k)
        if (!pats[k] || ms[k] < 7 || ms[k] > kHaloSmemMax)
            return fail(BMX_E_BADARG, "bmx_dict_create: pattern %d %s (every pattern: 7 <= m <= %d bytes)", k,
                        pats[k] ? "has a length outside that range" : "is NULL", kHaloSmemMax);
    if (int rc = check_device(device)) return rc;

    bmx_dict *d = new bmx_dict;
    d->device = device;
    d->npat = npat;
    d->sh = set_hash(npat, ms);
    d->slots_log2 = (uint32_t)kMultiSlotsLog2;
    while (((size_t)1 << d->slots_log2) < (size_t)8 * (size_t)npat) ++d->slots_log2;   // 4 entries per pattern, load <= 1/2
    d->occ_log2 = std::min<uint32_t>(d->slots_log2, (uint32_t)kDictMaxOccLog2);
    d->table_smem = d->slots_log2 <= (uint32_t)kDictMaxSmemSlotsLog2 ? 1u : 0u;
    const size_t slots = (size_t)1 << d->slots_log2, occ_bytes = ((size_t)1 << d->occ_log2) / 8;
    d->off_table = (size_t)kMultiBitmapWords * 4 + occ_bytes;
    d->off_dir = d->off_table + slots * 8;
    d->off_blob = d->off_dir + (((size_t)npat * 8 + 15) & ~size_t(15));
    d->blob_bytes = set_blob_bytes(npat, ms);
    std::vector<unsigned char> image(d->off_blob + d->blob_bytes + 16, 0);
    uint2 *table = reinterpret_cast<uint2 *>(image.data() + d->off_table);
    fill_set_tables(npat, pats, ms, d->sh, (int)d->slots_log2, reinterpret_cast<uint32_t *>(image.data()), table,
                    reinterpret_cast<uint2 *>(image.data() + d->off_dir), image.data() + d->off_blob);
    uint32_t *occ = reinterpret_cast<uint32_t *>(image.data() + (size_t)kMultiBitmapWords * 4);
    const size_t occ_mask = ((size_t)1 << d->occ_log2) - 1;
    for (size_t i = 0; i < slots; ++i)
        if (table[i].y != 0u) occ[(i & occ_mask) >> 5] |= 1u << (i & 31u);

    ScopedDevice keep;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void **>(&d->d_image), image.size());
    if (e == cudaSuccess) e = cudaMemcpy(d->d_image, image.data(), image.size(), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        bmx_dict_destroy(d);
        return fail(e == cudaErrorMemoryAllocation ? BMX_E_NOMEM : BMX_E_CUDA, "bmx_dict_create: %s", cudaGetErrorString(e));
    }
    *out = d;
    return BMX_OK;
}

void bmx_dict_destroy(bmx_dict *d)
{
    if (!d) return;
    if (d->d_image) {
        ScopedDevice keep;
        cudaSetDevice(d->device);
        cudaFree(d->d_image);
    }
    delete d;
}

int bmx_dict_search_device(const bmx_dict *d, const void *d_text, int64_t n, int64_t pos_base, int64_t *d_pos_out, int32_t *d_pat_out,
                           int64_t cap, uint64_t *counts, uint64_t *total_out, void *stream)
{
    if (int rc = check_search(d, d_text, n, d_pos_out, d_pat_out, cap, counts, total_out, "bmx_dict_search_device")) return rc;
    ThreadCtx *c = nullptr;
    if (int rc = get_ctx(d->device, &c)) return rc;
    return dict_search_resident(*c, d, static_cast<const unsigned char *>(d_text), n, pos_base, d_pos_out, d_pat_out,
                                d_pos_out ? cap : 0, counts, total_out, static_cast<cudaStream_t>(stream));
}

int bmx_dict_search(const bmx_dict *d, const char *text, int64_t n, int64_t *pos_out, int32_t *pat_out, int64_t cap, uint64_t *counts,
                    uint64_t *total_out)
{
    if (int rc = check_search(d, text, n, pos_out, pat_out, cap, counts, total_out, "bmx_dict_search")) return rc;
    ThreadCtx *c = nullptr;
    if (int rc = get_ctx(d->device, &c)) return rc;
    std::fill(counts, counts + d->npat, 0ull);
    *total_out = 0;
    if (n < d->sh.m_min) return BMX_OK;
    if (!pos_out) cap = 0;
    if (int rc = copy_text_resident(*c, text, n)) return rc;
    const unsigned char *d_text = static_cast<const unsigned char *>(c->text.p);
    cudaStream_t st = c->scan_stream;
    // device outputs in c.aux: a first guess of one pair per 64 bytes, grown to the total if the text is denser
    int64_t dcap = std::min<int64_t>(cap, first_pos_cap(n, d->sh.m_min, cap));
    for (int pass = 0; pass < 2; ++pass) {
        const size_t pat_off = ((size_t)dcap * 8 + 255) & ~size_t(255);
        if (int rc = ensure_buf(*c, c->aux, std::max<size_t>(pat_off + (size_t)dcap * 4, 256))) return rc;
        int64_t *d_pos = dcap > 0 ? static_cast<int64_t *>(c->aux.p) : nullptr;
        int32_t *d_pat = dcap > 0 ? reinterpret_cast<int32_t *>(static_cast<unsigned char *>(c->aux.p) + pat_off) : nullptr;
        if (int rc = dict_search_resident(*c, d, d_text, n, 0, d_pos, d_pat, dcap, counts, total_out, st)) return rc;
        const int64_t need = std::min<int64_t>((int64_t)*total_out, cap);
        if (need > dcap) {
            dcap = need;
            continue;
        }
        if (need > 0) {
            BMX_CUDA(cudaMemcpyAsync(pos_out, d_pos, (size_t)need * 8, cudaMemcpyDeviceToHost, st));
            BMX_CUDA(cudaMemcpyAsync(pat_out, d_pat, (size_t)need * 4, cudaMemcpyDeviceToHost, st));
            BMX_CUDA(cudaStreamSynchronize(st));
        }
        return BMX_OK;
    }
    return fail(BMX_E_CUDA, "bmx_dict_search: output buffers did not converge");
}

}  // extern "C"
