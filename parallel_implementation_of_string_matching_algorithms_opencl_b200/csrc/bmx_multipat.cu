// bmx_multipat.cu -- K patterns in ONE pass over the text (SURVEY 8f rank 3: multi-pattern batching).
//
// The reference builds its tables once per pattern (BoyreMoore/BoyreMoore/BoyreMoore.cpp:150-190) and would read
// the whole text again for every further pattern.  Here the text streams through shared memory once for all K:
//
//   filter   the same aligned q-gram hash as the single-pattern QGRAM filter, h = W[j] + hmul * W[j+1] (one gram
//            length q = min(12, m_min - 3) for all patterns; the third word joins for q > 8), but instead of 4 compares per pattern ONE probe of a
//            2^18-bit bitmap in shared memory ("some pattern has a gram with these top hash bits at some residue"):
//            the cost per text byte does not depend on K.
//   verify   flagged words (about 4K / 2^18 of them on random text) look their hash up in an exact table
//            {hash -> (pattern k, residue r)} and compare pattern k with the text at start = word - r.  Every match
//            bumps pattern k's counter (exact counts) and sets the start's bit in the UNION hit mask.
//   emit     the union masks go through the scanner's ordinary ordered emission (block scan + expand_kernel): an
//            ascending list U of the starts at which ANY pattern matches.
//   split    one CTA per pattern walks U, keeps the starts where its pattern matches (a comparison against the
//            text: U is short unless the text is dense) and writes them at their ranks: K ascending lists.
//
// Eligible: 1 <= K <= 64, every pattern 7 <= m <= 4096.  Anything else is searched pattern by pattern.
// Parity: each of the K results equals the serial reference result for that pattern alone (tests/: K serial
// oracle searches).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "bmx_ctx.h"

using namespace bmx;

namespace {

constexpr int kSplitThreads = 256;

struct MultiImage {
    std::vector<unsigned char> bytes;   // device image: [bitmap | table | dir | counts | split counts | out pointers | caps | blob]
    size_t off_table = 0, off_dir = 0, off_counts = 0, off_split = 0, off_out = 0, off_caps = 0, off_blob = 0;
    int32_t m_min = 0, m_max = 0;
    uint32_t hmul = 0, hmul2 = 0;
};

void build_multi_image(int32_t npat, const char *const *pats, const int32_t *ms, MultiImage *im)
{
    const SetHash sh = set_hash(npat, ms);
    im->m_min = sh.m_min;
    im->m_max = sh.m_max;
    im->hmul = sh.hmul;
    im->hmul2 = sh.hmul2;
    im->off_table = (size_t)kMultiBitmapWords * 4;
    im->off_dir = im->off_table + (size_t)kMultiSlots * 8;
    im->off_counts = im->off_dir + (size_t)kMultiMaxPatterns * 8;
    im->off_split = im->off_counts + (size_t)kMultiMaxPatterns * 8;
    im->off_out = im->off_split + (size_t)kMultiMaxPatterns * 8;
    im->off_caps = im->off_out + (size_t)kMultiMaxPatterns * 8;
    im->off_blob = im->off_caps + (size_t)kMultiMaxPatterns * 8;
    im->bytes.assign(im->off_blob + set_blob_bytes(npat, ms) + 16, 0);
    fill_set_tables(npat, pats, ms, sh, kMultiSlotsLog2, reinterpret_cast<uint32_t *>(im->bytes.data()),
                    reinterpret_cast<uint2 *>(im->bytes.data() + im->off_table), reinterpret_cast<uint2 *>(im->bytes.data() + im->off_dir),
                    im->bytes.data() + im->off_blob);
}

// One CTA per pattern: the starts of U at which pattern k matches, at their ranks.
__global__ void __launch_bounds__(kSplitThreads) multi_split_kernel(const int64_t *U, const unsigned long long *ucount, int64_t ucap,
                                                                    const uint8_t *text, int64_t n, const uint2 *dir, const uint8_t *blob,
                                                                    int64_t *const *out, const int64_t *caps, unsigned long long *split_counts)
{
    __shared__ uint32_t s_warp[kSplitThreads / 32];
    const int k = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint2 d = dir[k];
    const int32_t mk = (int32_t)d.y;
    const uint8_t *pk = blob + d.x;
    int64_t *dst = out[k];
    const int64_t cap = dst ? caps[k] : 0;
    const int64_t H = (int64_t)(*ucount < (unsigned long long)ucap ? *ucount : (unsigned long long)ucap);
    unsigned long long running = 0;
    for (int64_t base = 0; base < H; base += kSplitThreads) {
        const int64_t i = base + tid;
        int64_t p = 0;
        bool hit = false;
        if (i < H) {
            p = U[i];
            if (p + mk <= n) {
                hit = true;
                for (int32_t j = 0; hit && j < mk; ++j) hit = text[p + j] == pk[j];
            }
        }
        const uint32_t vote = __ballot_sync(0xFFFFFFFFu, hit);
        if (lane == 0) s_warp[warp] = __popc(vote);
        __syncthreads();
        uint32_t before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < kSplitThreads / 32; ++w) {
            const uint32_t c = s_warp[w];
            if (w < warp) before += c;
            total += c;
        }
        const unsigned long long rank = running + before + __popc(vote & ((1u << lane) - 1u));
        if (hit && (int64_t)rank < cap) dst[rank] = p;
        running += total;
        __syncthreads();
    }
    if (tid == 0) split_counts[k] = running;
}

}  // namespace

namespace bmx {

SetHash set_hash(int32_t npat, const int32_t *ms)
{
    SetHash sh;
    sh.m_min = *std::min_element(ms, ms + npat);
    sh.m_max = *std::max_element(ms, ms + npat);
    // one gram length for all patterns and residues: q = min(12, m_min - 3) bytes = 4 + q2 (second word) + q3 (third word)
    const int q = std::min(12, sh.m_min - 3);
    sh.q2 = std::min(4, q - 4);
    sh.q3 = std::max(0, q - 8);
    sh.hmul = gram_multiplier(kHashMul, sh.q2);
    sh.hmul2 = gram_multiplier(kHashMul2, sh.q3);
    return sh;
}

size_t set_blob_bytes(int32_t npat, const int32_t *ms)
{
    size_t blob = 0;
    for (int32_t k = 0; k < npat; ++k) blob += ((size_t)ms[k] + 8 + 15) & ~size_t(15);
    return blob;
}

void fill_set_tables(int32_t npat, const char *const *pats, const int32_t *ms, const SetHash &sh, int slots_log2, uint32_t *bits,
                     uint2 *table, uint2 *dir, unsigned char *blob)
{
    const uint32_t mask = (1u << slots_log2) - 1u;
    size_t at = 0;
    for (int32_t k = 0; k < npat; ++k) {
        const unsigned char *p = reinterpret_cast<const unsigned char *>(pats[k]);
        memcpy(blob + at, p, (size_t)ms[k]);
        dir[k] = make_uint2((uint32_t)at, (uint32_t)ms[k]);
        at += ((size_t)ms[k] + 8 + 15) & ~size_t(15);
        for (int r = 0; r < 4; ++r) {   // pattern byte r on a word boundary: the gram P[r .. r+q)
            const uint32_t h = set_gram_hash(sh, p + r);
            const uint32_t b = h >> (32 - kMultiBitmapLog2);
            bits[b >> 5] |= 1u << (b & 31u);
            uint32_t slot = (h * kMultiSlotMul) >> (32 - slots_log2);
            while (table[slot].y != 0u) slot = (slot + 1) & mask;
            table[slot] = make_uint2(h, 0x80000000u | ((uint32_t)k << 2) | (uint32_t)r);
        }
    }
}

// All K patterns over device-resident text d_text[0..n) in one pass (eligible sets only).  d_out[k] (device buffer of
// caps[k] entries, or NULL) receives pattern k's first min(counts[k], caps[k]) starts, ascending; counts[k] is exact.
int multi_scan_resident(ThreadCtx &c, const unsigned char *d_text, int64_t n, int32_t npat, const char *const *pats,
                        const int32_t *ms, int64_t *const *d_out, const int64_t *caps, uint64_t *counts, cudaStream_t st)
{
    MultiImage im;
    build_multi_image(npat, pats, ms, &im);
    for (int32_t k = 0; k < npat; ++k) counts[k] = 0;
    if (n < im.m_min) return BMX_OK;
    int64_t want = 0;
    bool any_out = false;
    for (int32_t k = 0; k < npat; ++k) {
        const int64_t ck = (d_out && d_out[k]) ? caps[k] : 0;
        reinterpret_cast<int64_t **>(im.bytes.data() + im.off_out)[k] = ck > 0 ? d_out[k] : nullptr;
        reinterpret_cast<int64_t *>(im.bytes.data() + im.off_caps)[k] = ck;
        any_out = any_out || ck > 0;
        want = std::min<int64_t>(n, want + std::min<int64_t>(ck, n));
    }
    if (int rc = ensure_buf(c, c.misc, im.bytes.size())) return rc;
    unsigned char *d_im = static_cast<unsigned char *>(c.misc.p);
    BMX_CUDA(cudaMemcpyAsync(d_im, im.bytes.data(), im.bytes.size(), cudaMemcpyHostToDevice, st));

    bmx_scanner *s = c.scanner;
    // the scanner leaves single-pattern mode: its cached pattern block no longer describes proto
    s->filter = kMulti;
    s->fold = false;
    s->pat.clear();
    s->proto = ScanArgs{};
    s->proto.m = im.m_min;
    s->proto.hmul = im.hmul;
    s->proto.hmul2 = im.hmul2;
    s->proto.g_mbits = reinterpret_cast<const uint32_t *>(d_im);
    s->proto.g_mtable = reinterpret_cast<const uint2 *>(d_im + im.off_table);
    s->proto.g_mdir = reinterpret_cast<const uint2 *>(d_im + im.off_dir);
    s->proto.g_mblob = d_im + im.off_blob;
    s->proto.mcounts = reinterpret_cast<unsigned long long *>(d_im + im.off_counts);
    s->proto.npat = (uint32_t)npat;
    const size_t blob_bytes = (im.bytes.size() - im.off_blob + 15) & ~size_t(15);
    s->proto.multi_blob_smem = blob_bytes <= (size_t)kPatSmemMax * 4 ? (uint32_t)blob_bytes : 0u;   // SmemCtl::good holds kPatSmemMax ints
    s->m = im.m_min;
    s->m_halo = im.m_max;
    ScopedTiming timing(s, 0);

    // from here on every failure breaks out of the loop, so that the scanner leaves multi-pattern mode below
    int64_t cap_u = any_out ? first_pos_room(c, n, im.m_min, want) : 0;
    std::vector<unsigned long long> h_counts((size_t)2 * kMultiMaxPatterns, 0);
    int rc = BMX_OK;
    for (int pass = 0; pass < 2 && rc == BMX_OK; ++pass) {
        if (cap_u > 0 && (rc = ensure_buf(c, c.pos, (size_t)cap_u * 8)) != BMX_OK) break;
        if (pass > 0 && cudaMemsetAsync(d_im + im.off_counts, 0, (size_t)kMultiMaxPatterns * 8, st) != cudaSuccess) {
            rc = fail(BMX_E_CUDA, "bmx_search_multi: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        int64_t *U = cap_u > 0 ? static_cast<int64_t *>(c.pos.p) : nullptr;
        if ((rc = bmx_scanner_begin(s, U, cap_u, st)) != BMX_OK) break;
        if ((rc = bmx_scanner_scan(s, d_text, n, 0, st)) != BMX_OK) break;
        if (U) {
            multi_split_kernel<<<npat, kSplitThreads, 0, st>>>(U, result_slot(s), cap_u, d_text, n, s->proto.g_mdir, s->proto.g_mblob,
                                                                reinterpret_cast<int64_t *const *>(d_im + im.off_out),
                                                                reinterpret_cast<const int64_t *>(d_im + im.off_caps),
                                                                reinterpret_cast<unsigned long long *>(d_im + im.off_split));
            if (cudaGetLastError() != cudaSuccess) {
                rc = fail(BMX_E_CUDA, "multi_split launch failed");
                break;
            }
        }
        if (cudaMemcpyAsync(h_counts.data(), d_im + im.off_counts, (size_t)2 * kMultiMaxPatterns * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess) {
            rc = fail(BMX_E_CUDA, "bmx_search_multi: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        uint64_t ucount = 0;
        if ((rc = bmx_scanner_finish(s, &ucount, nullptr, st)) != BMX_OK) break;   // synchronises st
        bool short_list = false;
        for (int32_t k = 0; k < npat && U; ++k) {
            const int64_t ck = reinterpret_cast<const int64_t *>(im.bytes.data() + im.off_caps)[k];
            if ((int64_t)h_counts[(size_t)kMultiMaxPatterns + k] < std::min<int64_t>(ck, (int64_t)h_counts[(size_t)k])) short_list = true;
        }
        if (!short_list || (int64_t)ucount <= cap_u) break;
        cap_u = (int64_t)ucount;   // the union list was cut short before some pattern had its share: room for all of it
    }
    s->m_halo = 0;
    s->m = 0;   // the scanner has no single pattern until the next set_pattern
    if (rc != BMX_OK) return rc;
    for (int32_t k = 0; k < npat; ++k) counts[k] = h_counts[(size_t)k];
    return BMX_OK;
}

bool multi_eligible(int32_t npat, const int32_t *ms)
{
    if (npat < 1 || npat > kMultiMaxPatterns) return false;
    for (int32_t k = 0; k < npat; ++k)
        if (ms[k] < 7 || ms[k] > kHaloSmemMax) return false;
    return true;
}

}  // namespace bmx

extern "C" {

int bmx_search_multi_device(const void *d_text, int64_t n, int32_t npat, const char *const *pats, const int32_t *ms,
                            int64_t *const *d_pos_out, const int64_t *pos_cap, uint64_t *counts, void *stream)
{
    if (int rc = check_text(d_text, n, "bmx_search_multi_device")) return rc;
    if (int rc = check_pattern_set(npat, pats, ms, d_pos_out, pos_cap, counts, "bmx_search_multi_device")) return rc;
    if (npat == 0 || n == 0) return BMX_OK;
    ThreadCtx *c = nullptr;
    if (int rc = current_ctx(&c)) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (multi_eligible(npat, ms))
        return multi_scan_resident(*c, static_cast<const unsigned char *>(d_text), n, npat, pats, ms, d_pos_out, pos_cap, counts, st);
    // not eligible for the shared table (a pattern shorter than 7 or longer than 4096 bytes, or more than 64 patterns):
    // one pass per pattern over the resident text
    for (int32_t k = 0; k < npat; ++k) {
        if (n < ms[k]) continue;
        int64_t *out = d_pos_out ? d_pos_out[k] : nullptr;
        if (int rc = search_once(c->scanner, pats[k], ms[k], BMX_VARIANT_AUTO, d_text, n, 0, out, out ? pos_cap[k] : 0, &counts[k], nullptr, st))
            return rc;
    }
    return BMX_OK;
}

}  // extern "C"
