// bmx_scan.cu -- the sm_100a scan kernels of libbmx.so and their launch planning.
//
// Replaces the device side of the reference's hot path: the OpenCL kernel `search`
// (BoyreMoore/x64/Debug/kernel1.cl:1-35, launched with global=2, local=1 from
// BoyreMoore/BoyreMoore/BoyreMoore.cpp:273-280).  The reference walks each partition with ONE
// work-item, one dependent byte load at a time.  Here the text streams through shared memory
// exactly once:
//
//   producer warp   one elected lane claims tiles from a global ticket counter and stages
//                   [16 B pre | TILE | halo] of text per tile into a ring of shared-memory
//                   stages with 1-D TMA bulk copies (cp.async.bulk ... mbarrier::complete_tx).
//   consumer warps  8 warps read the stage with 16-byte LDS.128, run a branch-free candidate
//                   filter over 16 start positions per thread and vote with __ballot_sync; a chunk
//                   with candidates is then checked by the whole warp at once (coop_verify16:
//                   16 start positions x 2 pattern words per ballot).  Patterns that do not fit
//                   shared memory (m > 1024) are verified by the flagged lanes right-to-left with
//                   the reference's bad-symbol / good-suffix shifts (kernel1.cl:21-33) pruning
//                   their own candidate bits (verify_candidates).
//   emission        every thread holds a 16-bit hit mask per 16-byte chunk.  Warps whose 2 KiB
//                   segment has hits store the masks (mask16) and the segment's hit count
//                   (seg_count, block_sum); no CTA ever waits for another one.  The CTA
//                   that finishes last turns the per-2-MiB block sums into exclusive bases, and
//                   expand_kernel (one warp per 32 KiB item) re-derives each segment's rank and
//                   writes every hit at its exact rank with coalesced stores.  Ranks are
//                   exact prefix sums, so the list is ascending and bit-identical from run to
//                   run regardless of scheduling.
//
// Filters (bmx_variant):
//   QGRAM    m >= 7.  Any occurrence covers the aligned 32-bit word at ceil(p/4)*4 and the word
//            after it; h = W[j] + hmul * W[j+1] is compared with the 4 pattern hashes for
//            r = (4 - p%4)%4.  1 IMAD + 4 ISETP per 4 text bytes, no funnel shifts.
//   WINDOW   any m.  m >= 4: the 4-byte window at every position (funnel shifts) against P[0..4), exact
//            for m = 4.  m <= 3, and m = 5, 6 on small alphabets: four start positions per word at once
//            (zero-byte detection over the XOR with the replicated pattern bytes), exact up to five bytes.
//   SHIFTAND m <= 32. Bit-parallel Shift-And (the Shift-Or family): D = ((D<<1)|1) & B[c].
//            Kept because the north star asks for the comparison; measured slower (DESIGN.md).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <utility>

#include "bmx_ctx.h"

namespace bmx {

// ---------------------------------------------------------------------------------------------
// PTX helpers: mbarrier, 1-D TMA bulk copy
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
// (A suspend-time hint on try_wait was measured neutral on sparse and mid-density texts alike and is not used.)
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "BMX_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra BMX_DONE_%=;\n"
        "bra BMX_WAIT_%=;\n"
        "BMX_DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// global -> shared bulk copy (TMA, 1-D): bytes % 16 == 0, both addresses 16-byte aligned.
__device__ __forceinline__ void tma_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    // the text is streamed exactly once: mark its lines evict-first so they do not push the emission
    // scratch (segment counts, masks) out of L2
    uint64_t policy;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
                 : "memory");
}
// Barrier over the consumer threads only (the producer warp has its own life cycle).
__device__ __forceinline__ void bar_sync_consumers()
{
    asm volatile("barrier.cta.sync 1, %0;" ::"r"(kConsumerThreads) : "memory");
}
// ASCII case fold of four bytes at once ('A'..'Z' -> 'a'..'z', every other byte value unchanged): for a byte b < 0x80,
// t + 0x3F reaches bit 7 iff b >= 'A' and t + 0x25 iff b > 'Z'; t <= 0x7F, so no sum carries into the next byte.
__device__ __forceinline__ uint32_t fold_word(uint32_t w)
{
    const uint32_t t = w & 0x7F7F7F7Fu;
    const uint32_t u = (t + 0x3F3F3F3Fu) & ~(t + 0x25252525u) & ~w & 0x80808080u;
    return w | (u >> 2);
}
// Case-insensitive scans fold a whole stage ([16 B pre | tile | halo]) in place, once, before any warp reads it, so
// every reader of the stage (filters, coop_verify16, verify_candidates, dense_tile, Shift-And) sees folded text.
// The stores are generic-proxy writes to memory the next TMA copy (async proxy) overwrites: each thread orders its
// stores before that copy with a proxy fence, ahead of its warp's arrival on empty[s].
__device__ __forceinline__ void fold_stage(uint8_t *stage, uint32_t bytes, int tid)
{
    uint4 *p = reinterpret_cast<uint4 *>(stage);
#pragma unroll 4
    for (uint32_t i = (uint32_t)tid; i < bytes / 16u; i += kConsumerThreads) {
        uint4 v = p[i];
        v.x = fold_word(v.x);
        v.y = fold_word(v.y);
        v.z = fold_word(v.z);
        v.w = fold_word(v.w);
        p[i] = v;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// ---------------------------------------------------------------------------------------------
// Shared-memory control block (the stages follow it, 128-byte aligned)
// ---------------------------------------------------------------------------------------------
struct SmemCtl {
    uint64_t full[kMaxStages];     // producer -> consumers: tile bytes have landed
    uint64_t empty[kMaxStages];    // consumers -> producer: stage may be overwritten
    int32_t slot_tile[kMaxStages]; // tile index staged in each slot, -1 = no more tiles
    uint32_t is_last;              // this CTA finished last: it scans the block sums
    unsigned long long scan_warp[kConsumerWarps];
    uint32_t scan_dense[kConsumerWarps];
    int32_t bad[256];              // bad-symbol table   (BoyreMoore.cpp:153-162)
    uint32_t sa_mask[256];         // Shift-And occurrence masks
    alignas(16) int32_t good[kPatSmemMax];  // good-suffix table  (BoyreMoore.cpp:165-190); the multi-pattern variant keeps its patterns here
    uint8_t pat[kPatSmemMax];
    uint32_t rpat[kPatSmemMax / 4];  // pattern words from the right end: rpat[i] = P[m-4-4i .. m-4i), little endian
};
constexpr size_t kCtlBytes = (sizeof(SmemCtl) + 127) & ~size_t(127);

// ---------------------------------------------------------------------------------------------
// Candidate verification with Boyer-Moore skips
// ---------------------------------------------------------------------------------------------
// cand: candidate bits (bit b = start position p0 + b).  text(v) = vbase[v].  Follows the
// reference loop (kernel1.cl:19-34): compare right to left; on a match record the start and
// advance by one (:24); on a mismatch after k matched bytes advance by d1 = max(bad[T[i]]-k, 1)
// (T[i] = byte under the LAST pattern position, :27-28) or max(d1, good[k]) when k > 0
// (:29-31).  "Advance" here means: candidate bits inside the skipped range are dropped.
// 4 bytes at byte offset `off` from a 4-byte aligned base (shared, global or generic memory), little endian.
__device__ __forceinline__ uint32_t load_u32_unaligned(const uint8_t *base, int64_t off)
{
    const uint32_t *w = reinterpret_cast<const uint32_t *>(base + (off & ~int64_t(3)));
    return __funnelshift_r(w[0], w[1], 8 * (int)(off & 3));
}

// `wordwise` is set when the text is verified from the staged tile (whose halo makes the aligned word
// pairs safe to read); long patterns verified from global memory compare byte by byte.
// `rpat` (shared memory, patterns up to kPatSmemMax bytes): the pattern's words counted from its right end.  With it
// a step of the right-to-left comparison is ONE new aligned text word (the previous one is kept for the funnel shift),
// one pattern word and an XOR -- a 25-byte match costs ~60 instructions instead of ~220 with two unaligned word
// fetches (four loads, two shifts, 64-bit address arithmetic) per step.
// cand holds the candidates of ALL FOUR slabs of the lane's share of a segment (16 bits each, slab sl at bits 16 sl ..):
// one call per segment instead of one per slab -- candidates of different slabs usually sit in different lanes, and
// lanes of one call verify concurrently, so a segment with candidates in three slabs pays for one verification, not three.
// FOLD (case-insensitive scans): the pattern and tables are folded, and so is a staged tile, but text read from global
// memory (m > kHaloSmemMax) is the caller's: its bytes are folded as they are compared and looked up in bad[].
template <bool FOLD>
__device__ __noinline__ unsigned long long verify_candidates(unsigned long long cand, const uint8_t *vbase, int64_t p0, int32_t m,
                                                             const uint8_t *pat, const uint32_t *rpat, const int32_t *bad,
                                                             const int32_t *good, bool wordwise)
{
    auto tb = [](uint8_t c) -> uint8_t { return FOLD && (uint32_t)(c - 'A') < 26u ? (uint8_t)(c | 0x20u) : c; };
    unsigned long long hits = 0;
    while (cand) {
        const int b = __ffsll((long long)cand) - 1;
        const int64_t p = p0 + (b >> 4) * 512 + (b & 15);   // slab b / 16 starts 512 bytes behind the previous one
        const uint8_t *t = vbase + p;
        // k = number of pattern bytes that match from the right end (kernel1.cl:21-22), found four
        // bytes at a time: in a little-endian word the rightmost text byte is the most significant one,
        // so the leading zero bytes of the XOR are exactly the matched suffix bytes of that word.
        int32_t k = 0;
        bool differs = false;
        if (wordwise && rpat != nullptr) {
            const uintptr_t end = reinterpret_cast<uintptr_t>(t) + (uintptr_t)m;      // one past the last text byte
            const uint32_t *aw = reinterpret_cast<const uint32_t *>(end & ~uintptr_t(3));
            const int sh = 8 * (int)(end & 3u);
            uint32_t hi = aw[0];          // the word holding the byte behind the window: inside the staged halo
            const int32_t steps = m >> 2;
            for (int32_t i = 0; i < steps; ++i) {
                const uint32_t lo = *--aw;
                const uint32_t x = __funnelshift_r(lo, hi, sh) ^ rpat[i];   // text bytes [m-4-4i, m-4i) of the window
                hi = lo;
                if (x) {
                    k += __clz(x) >> 3;
                    differs = true;
                    break;
                }
                k += 4;
            }
        } else {
            while (wordwise && k + 4 <= m) {
                const uint32_t x = load_u32_unaligned(vbase, p + m - 4 - k) ^ load_u32_unaligned(pat, m - 4 - k);
                if (x) {
                    k += __clz(x) >> 3;
                    differs = true;
                    break;
                }
                k += 4;
            }
        }
        if (!differs)
            while (k < m && tb(t[m - 1 - k]) == pat[m - 1 - k]) ++k;
        int32_t shift;
        if (k == m) {
            hits |= 1ull << b;
            shift = 1;
        } else {
            int32_t d1 = bad[tb(t[m - 1])] - k;
            d1 = d1 > 1 ? d1 : 1;
            shift = d1;
            if (k > 0) {
                const int32_t d2 = good[k];
                shift = d2 > d1 ? d2 : d1;
            }
        }
        // the shift skips candidates of THIS slab only (the next slab's start positions lie 512 bytes further on)
        const int in_slab = (b & 15) + shift;
        const int nb = in_slab >= 16 ? (b | 15) + 1 : b + shift;
        cand = nb >= 64 ? 0ull : ((cand >> nb) << nb);
    }
    return hits;
}

// Warp-cooperative exact check of the 16 start positions owned by one 16-byte chunk -- what the sparse path does with
// a chunk the filter flagged.  The walk above is one lane following the reference's loop while 31 lanes wait, a chain
// of dependent shared-memory loads per candidate; here the whole warp looks at the chunk at once: lane i compares one
// of the pattern's LAST two words at start position (i & 15) -- the filter's q-gram sits at the pattern's front, so the
// tail is what tells "occurrences starting from" from "occurrences by process" --, one ballot keeps the positions whose
// last 8 bytes match, and each survivor (almost always a true occurrence) has the words in front compared 32 words =
// 128 bytes per step.  The result is the same set the reference's loop reports -- it advances by one after a match
// (kernel1.cl:24), so every occurrence is reported; the skips only prune non-matches.
// Everything that depends only on the lane is computed once per kernel (CoopLane): a chunk starts on a 16-byte
// boundary, so the aligned word a lane reads, its funnel shift and its (masked) pattern word never change.
struct CoopLane {
    int32_t off1;     // phase 1: byte offset (multiple of 4, may be -4) of the lane's aligned word pair from the chunk
    uint32_t sh1;     //          funnel shift in bits
    uint32_t pw1, pm1;  //        the lane's pattern word (one of the last two) and its byte mask (0: the pattern has no such word)
    uint32_t pw2, pm2;  // phase 2, first round: pattern word `lane` (in front of the last two) and its mask
    int32_t nwords, front;   // pattern words; words in front of the last two
};
__device__ __forceinline__ uint32_t pat_word_mask(int32_t wi, int32_t m)
{
    const int32_t left = m - 4 * wi;   // pattern bytes in word wi
    return left >= 4 ? 0xFFFFFFFFu : (left <= 0 ? 0u : (0xFFFFFFFFu >> (32 - 8 * left)));
}
template <int OFFS>
__device__ __forceinline__ CoopLane coop_lane_setup(const uint32_t *patw, int32_t m, int lane)
{
    CoopLane c;
    c.nwords = (m + 3) >> 2;
    c.front = c.nwords > 2 ? c.nwords - 2 : 0;
    const int32_t w1 = c.front + (lane >> 4);
    const int32_t o1 = OFFS + (lane & 15) + 4 * w1;
    c.off1 = o1 & ~3;
    c.sh1 = 8u * (uint32_t)(o1 & 3);
    c.pm1 = pat_word_mask(w1, m);
    c.pw1 = c.pm1 ? patw[w1] & c.pm1 : 0u;
    c.pm2 = lane < c.front ? 0xFFFFFFFFu : 0u;
    c.pw2 = c.pm2 ? patw[lane] : 0u;
    return c;
}
// cp: first byte of the chunk in the staged tile (16-byte aligned).  Returns the hit bits of the chunk (bit b = start
// position cp + OFFS + b).
template <int OFFS>
__device__ __forceinline__ uint32_t coop_verify16(const uint8_t *cp, const CoopLane &c, const uint32_t *patw, int lane)
{
    const uint32_t *w1 = reinterpret_cast<const uint32_t *>(cp + c.off1);
    const uint32_t x1 = __funnelshift_r(w1[0], w1[1], c.sh1);
    const uint32_t b = __ballot_sync(0xFFFFFFFFu, ((x1 ^ c.pw1) & c.pm1) == 0u);
    uint32_t alive = b & (b >> 16);
    if (c.front > 0) {
        uint32_t left = alive;
        while (left) {
            const int32_t bit = __ffs(left) - 1;
            left &= left - 1;
            // word `lane` of the pattern at start position OFFS + bit: the alignment is the same for all lanes
            const int32_t o2 = OFFS + bit;
            const uint32_t *w2 = reinterpret_cast<const uint32_t *>(cp + (o2 & ~3)) + lane;
            const uint32_t sh2 = 8u * (uint32_t)(o2 & 3);
            // (lanes beyond the pattern's words load nothing: their words may lie behind the staged halo)
            uint32_t x2 = 0u;
            if (c.pm2) x2 = __funnelshift_r(w2[0], w2[1], sh2);
            bool same = __all_sync(0xFFFFFFFFu, ((x2 ^ c.pw2) & c.pm2) == 0u);
            for (int32_t w0 = 32; w0 < c.front && same; w0 += 32) {   // patterns longer than 136 bytes
                const int32_t wi = w0 + lane;
                uint32_t x = 0u, pw = 0u;
                if (wi < c.front) {
                    x = __funnelshift_r(w2[w0], w2[w0 + 1], sh2);
                    pw = patw[wi];
                }
                same = __all_sync(0xFFFFFFFFu, x == pw);
            }
            if (!same) alive &= ~(1u << bit);
        }
    }
    return alive;
}

// Bits b (0..15) whose start position p0 + b lies in [vmin, vmax].
__device__ __forceinline__ uint32_t valid_bits(int64_t p0, int64_t vmin, int64_t vmax)
{
    const int64_t lo = vmin - p0, hi = vmax - p0;
    if (hi < 0 || lo > 15) return 0u;
    const uint32_t mlo = lo <= 0 ? 0xFFFFu : ((0xFFFFu << (int)lo) & 0xFFFFu);
    const uint32_t mhi = hi >= 15 ? 0xFFFFu : (0xFFFFu >> (15 - (int)hi));
    return mlo & mhi;
}

// ---------------------------------------------------------------------------------------------
// The scan kernel
// ---------------------------------------------------------------------------------------------
// WINDOW: the 4-byte window that starts s bytes into `lo` (continuing in `hi`).  (Building the
// shifted windows on the FMA pipe with IMAD.HI/IMAD instead of SHF was measured 13 % slower.)
__device__ __forceinline__ uint32_t window_at(uint32_t lo, uint32_t hi, int s)
{
    return s == 0 ? lo : __funnelshift_r(lo, hi, 8 * s);
}

// WINDOW, m <= 3: four start positions per word at once.  z = OR over k of ((text shifted by k bytes) ^ P[k] in every
// byte) has a zero byte exactly where all m bytes match; (z & 0x7F..) + 0x7F.. never carries across bytes, so the zero
// test is exact.  Returns 0x80 in the byte of every matching start position: 3 + 2(m-1) + 3 instructions for four
// positions instead of a funnel shift, a multiply, a compare and a select each.
template <int M>   // M = bytes tested, 1..5: a compile-time constant, so the construction below is branch-free
__device__ __forceinline__ uint32_t window_flags(uint32_t lo, uint32_t hi, uint32_t b0, uint32_t b1, uint32_t b2, uint32_t b3 = 0u, uint32_t b4 = 0u)
{
    uint32_t z = lo ^ b0;
    if (M >= 2) z |= __funnelshift_r(lo, hi, 8) ^ b1;
    if (M >= 3) z |= __funnelshift_r(lo, hi, 16) ^ b2;
    if (M >= 4) z |= __funnelshift_r(lo, hi, 24) ^ b3;
    if (M >= 5) z |= hi ^ b4;   // the byte four positions on is the same byte of the next word
    const uint32_t a = (z & 0x7F7F7F7Fu) + 0x7F7F7F7Fu;
    return ~(a | z) & 0x80808080u;
}

template <Filter F>
__device__ __forceinline__ bool filter_any(const uint4 &w, uint32_t w4, const ScanArgs &A)
{
    if (filter_variant(F) == BMX_VARIANT_QGRAM) {
        const uint32_t f0 = A.f[0], f1 = A.f[1], f2 = A.f[2], f3 = A.f[3];
        // hmul = K << (32 - 8*q2): the multiplication itself drops the bytes of the second word that lie
        // beyond the q-gram (7 <= m <= 10), so short patterns need no masking instruction
        if (F == kQgramPerResidue) {
            // 7 <= m <= 10: residue r may use min(8, m - r) pattern bytes, so each residue hashes with its
            // own multiplier -- 3 more IMADs per word, several times fewer candidates on small alphabets
            const uint32_t k0 = A.hmulr[0], k1 = A.hmulr[1], k2 = A.hmulr[2], k3 = A.hmulr[3];
            const uint32_t ww[5] = {w.x, w.y, w.z, w.w, w4};
            bool any = false;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                any |= (ww[j] + k0 * ww[j + 1] == f0) | (ww[j] + k1 * ww[j + 1] == f1);
                any |= (ww[j] + k2 * ww[j + 1] == f2) | (ww[j] + k3 * ww[j + 1] == f3);
            }
            return any;
        }
        const uint32_t km = A.hmul;
        const uint32_t h0 = w.x + km * w.y;
        const uint32_t h1 = w.y + km * w.z;
        const uint32_t h2 = w.z + km * w.w;
        const uint32_t h3 = w.w + km * w4;
        bool any = (h0 == f0) | (h0 == f1) | (h0 == f2) | (h0 == f3);
        any |= (h1 == f0) | (h1 == f1) | (h1 == f2) | (h1 == f3);
        any |= (h2 == f0) | (h2 == f1) | (h2 == f2) | (h2 == f3);
        any |= (h3 == f0) | (h3 == f1) | (h3 == f2) | (h3 == f3);
        return any;
    } else {
        if constexpr (filter_bytes(F) != 0) {   // m <= 3, or the first five bytes of a 5- or 6-byte pattern
            constexpr int M = filter_bytes(F);
            const uint32_t b0 = A.bcast[0], b1 = A.bcast[1], b2 = A.bcast[2], b3 = A.bcast[3], b4 = A.bcast[4];
            return (window_flags<M>(w.x, w.y, b0, b1, b2, b3, b4) | window_flags<M>(w.y, w.z, b0, b1, b2, b3, b4) |
                    window_flags<M>(w.z, w.w, b0, b1, b2, b3, b4) | window_flags<M>(w.w, w4, b0, b1, b2, b3, b4)) != 0u;
        }
        const uint32_t tg = A.f[0];
        const uint32_t ww[5] = {w.x, w.y, w.z, w.w, w4};
        bool any = false;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
            for (int sh = 0; sh < 4; ++sh) any |= window_at(ww[j], ww[j + 1], sh) == tg;
        }
        return any;
    }
}

template <Filter F>
__device__ __forceinline__ uint32_t filter_mask(const uint4 &w, uint32_t w4, const ScanArgs &A)
{
    uint32_t mask = 0;
    const uint32_t ww[5] = {w.x, w.y, w.z, w.w, w4};
    if (filter_variant(F) == BMX_VARIANT_QGRAM) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t h = ww[j] + A.hmul * ww[j + 1];
            // word j with residue r flags start position 4j - r, i.e. bit 4j + 3 - r (bit 0 = c - 3)
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const uint32_t hr = F == kQgram ? h : ww[j] + A.hmulr[r] * ww[j + 1];
                mask |= (uint32_t)(hr == A.f[r]) << (4 * j + 3 - r);
            }
        }
    } else if constexpr (filter_bytes(F) != 0) {
        // flags of two words share one multiply that gathers their eight 0x80 bits into one byte
        // ((c0 >> 4 | c1) * 0x204081 >> 24: bits 3,11,19,27 and 7,15,23,31 land on 24..31 in position order, no carries)
        constexpr int M = filter_bytes(F);
        const uint32_t b0 = A.bcast[0], b1 = A.bcast[1], b2 = A.bcast[2], b3 = A.bcast[3], b4 = A.bcast[4];
        const uint32_t c0 = window_flags<M>(ww[0], ww[1], b0, b1, b2, b3, b4), c1 = window_flags<M>(ww[1], ww[2], b0, b1, b2, b3, b4);
        const uint32_t c2 = window_flags<M>(ww[2], ww[3], b0, b1, b2, b3, b4), c3 = window_flags<M>(ww[3], ww[4], b0, b1, b2, b3, b4);
        mask = ((((c0 >> 4) | c1) * 0x00204081u) >> 24) | (((((c2 >> 4) | c3) * 0x00204081u) >> 24) << 8);
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
            for (int sh = 0; sh < 4; ++sh) mask |= (uint32_t)(window_at(ww[j], ww[j + 1], sh) == A.f[0]) << (4 * j + sh);
        }
    }
    return mask;
}

// Shift-And over one thread's 16 start positions: bytes tp[0 .. 16+m-2].
__device__ __forceinline__ uint32_t shiftand_chunk(const uint8_t *tp, int32_t m, const uint32_t *sa_mask)
{
    uint32_t D = 0, hits = 0;
    const int total = 16 + m - 1;
    const uint32_t top = m - 1;
    for (int u = 0; u < total; u += 16) {
        const uint4 q = *reinterpret_cast<const uint4 *>(tp + u);
        const uint32_t ww[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const int v = u + 4 * j + s;
                const uint32_t c = (ww[j] >> (8 * s)) & 0xFFu;
                D = ((D << 1) | 1u) & sa_mask[c];
                const int start = v - (int)top;  // start position of a match ending at byte v
                if (start >= 0 && start < 16) hits |= ((D >> top) & 1u) << start;
            }
        }
    }
    return hits;
}

// ---- multi-pattern variant: one probe per aligned word, independent of the number of patterns ---------------
// h = W[j] + hmul * W[j+1] as in QGRAM (one gram length for all patterns); bit (h >> 14) of a 2^18-bit bitmap in
// shared memory says "some pattern has a q-gram with these top hash bits at some residue".  Only flagged words
// go on to the exact table {hash -> (pattern, residue)} and from there to a plain comparison with that pattern.
struct MultiSmem {
    const uint32_t *bits;
    const uint2 *table;
    const uint2 *dir;
    const uint32_t *occ;   // kDict: "home slot occupied", folded to 2^mocc_log2 bits (may say occupied wrongly, never empty)
};
__device__ __forceinline__ uint32_t multi_probe(const uint32_t *bits, uint32_t h)
{
    return __funnelshift_r(bits[h >> (32 - kMultiBitmapLog2 + 5)], 0u, h >> (32 - kMultiBitmapLog2));  // bit 0 = the flag
}
__device__ __forceinline__ bool multi_any(const uint4 &w, uint32_t w4, uint32_t w5, uint32_t k1, uint32_t k2, const uint32_t *bits)
{
    // grams of up to 12 bytes: the third word joins the hash when every pattern is long enough (k2 != 0), which is
    // what keeps small alphabets selective (4^-12 instead of 4^-8 per gram on DNA)
    const uint32_t f = multi_probe(bits, w.x + k1 * w.y + k2 * w.z) | multi_probe(bits, w.y + k1 * w.z + k2 * w.w) |
                       multi_probe(bits, w.z + k1 * w.w + k2 * w4) | multi_probe(bits, w.w + k1 * w4 + k2 * w5);
    return (f & 1u) != 0u;
}
// A word whose hash is flagged AND whose home slot of the exact table is occupied: walk the probe sequence and compare
// the text with every pattern that has this gram at some residue.  Rare (about K / 128 of the flagged words), out of
// line, all arguments in registers.  Returns the hit bits of the chunk (bit = start - (chunk_v - 3)).
// kMulti's table has kMultiSlots slots; a dictionary's (kDict) has 2^mslots_log2, in shared or global memory.
template <Filter F>
__device__ __noinline__ uint32_t multi_word(const ScanArgs &A, const uint2 *table, const uint2 *dir, const uint8_t *blob,
                                            uint32_t h, int j, int64_t chunk_v, const uint8_t *vbase)
{
    const uint32_t lg = F == kMulti ? (uint32_t)kMultiSlotsLog2 : A.mslots_log2, mask = (1u << lg) - 1u;
    uint32_t hits = 0;
    for (uint32_t slot = (h * kMultiSlotMul) >> (32 - lg);; slot = (slot + 1) & mask) {
        const uint2 e = table[slot];
        if (e.y == 0u) break;
        if (e.x != h) continue;
        const uint32_t k = (e.y >> 2) & 0xFFFFu, r = e.y & 3u;
        const uint2 d = dir[k];
        const int32_t mk = (int32_t)d.y;
        const int64_t p = chunk_v + 4 * j - (int64_t)r;
        if (p < A.vmin || p > A.vmax || p + mk > A.vlen) continue;
        const uint8_t *pk = blob + d.x;
        bool same = true;
        int32_t i = 0;
        for (; same && i + 4 <= mk; i += 4) same = load_u32_unaligned(vbase, p + i) == *reinterpret_cast<const uint32_t *>(pk + i);
        for (; same && i < mk; ++i) same = vbase[p + i] == pk[i];
        if (same) {
            hits |= 1u << (4 * j + 3 - (int)r);
            atomicAdd(A.mcounts + k, 1ull);
        }
    }
    return hits;
}
// Exact check of one 16-byte chunk (start positions c-3 .. c+12, c = chunk_v): returns the union hit mask and bumps the
// per-pattern counters.  Every start position is examined by exactly one thread of the grid.  A false positive of the
// bitmap dies here at ONE shared-memory load (its home slot in the exact table is empty), without a call; a dictionary
// whose table is too large for shared memory asks the staged occupancy bits instead of the table.
template <Filter F>
__device__ __forceinline__ uint32_t multi_chunk(const ScanArgs &A, const MultiSmem &M, const uint8_t *blob, const uint4 &w, uint32_t w4,
                                                uint32_t w5, int64_t chunk_v, const uint8_t *vbase)
{
    const uint32_t k1 = A.hmul, k2 = A.hmul2;
    const uint32_t h[4] = {w.x + k1 * w.y + k2 * w.z, w.y + k1 * w.z + k2 * w.w, w.z + k1 * w.w + k2 * w4, w.w + k1 * w4 + k2 * w5};
    uint32_t hits = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (!(multi_probe(M.bits, h[j]) & 1u)) continue;
        bool home;
        if constexpr (F == kMulti) {
            home = M.table[(h[j] * kMultiSlotMul) >> (32 - kMultiSlotsLog2)].y != 0u;
        } else {
            const uint32_t b = ((h[j] * kMultiSlotMul) >> (32 - A.mslots_log2)) & ((1u << A.mocc_log2) - 1u);
            home = (M.occ[b >> 5] >> (b & 31u)) & 1u;
        }
        if (home) hits |= multi_word<F>(A, M.table, M.dir, blob, h[j], j, chunk_v, vbase);
    }
    return hits;
}

// The second word after each chunk (three-word grams of the multi-pattern variant), same rotation as w4.
__device__ __forceinline__ void load_second_after(const uint8_t *sp, int lane, const uint4 (&w)[4], uint32_t (&w5)[4])
{
    const uint32_t after2 = *reinterpret_cast<const uint32_t *>(sp + kSegBytes + 4);  // broadcast load
#pragma unroll
    for (int sl = 0; sl < 4; ++sl) {
        const uint32_t wrap = sl < 3 ? w[sl < 3 ? sl + 1 : 3].y : after2;
        w5[sl] = __shfl_sync(0xFFFFFFFFu, lane == 0 ? wrap : w[sl].y, (lane + 1) & 31);
    }
}

__device__ __forceinline__ void load_segment(const uint8_t *sp, int lane, uint4 (&w)[4], uint32_t (&w4)[4])
{
#pragma unroll
    for (int sl = 0; sl < 4; ++sl) w[sl] = *reinterpret_cast<const uint4 *>(sp + sl * 512 + lane * 16);
    const uint32_t after = *reinterpret_cast<const uint32_t *>(sp + kSegBytes);  // broadcast load
#pragma unroll
    for (int sl = 0; sl < 4; ++sl) {
        const uint32_t wrap = sl < 3 ? w[sl < 3 ? sl + 1 : 3].x : after;
        w4[sl] = __shfl_sync(0xFFFFFFFFu, lane == 0 ? wrap : w[sl].x, (lane + 1) & 31);
    }
}

// A warp whose segment has hits publishes its masks and its count (no waiting on anyone) and returns
// the segment's hit count; the caller adds a warp's counts of one tile to the block sum in one atomic
// (the per-segment atomics of an every-segment-hits text queued up on a handful of L2 addresses).
__device__ __forceinline__ uint32_t publish_segment(const ScanArgs &A, uint32_t seg, const uint32_t (&hm)[4],
                                                    uint32_t seg_hits, int lane)
{
    const uint32_t total = __reduce_add_sync(0xFFFFFFFFu, seg_hits);  // REDUX.SUM
    if (total != kSegBytes) {  // a full segment (every start matches) needs no masks
        uint16_t *mk = A.mask16 + (size_t)seg * kSegChunks + lane;
#pragma unroll
        for (int sl = 0; sl < 4; ++sl) mk[sl * 32] = (uint16_t)hm[sl];
    }
    if (lane == 0) {
        A.seg_count[seg] = (uint16_t)total;
        A.item_flag[seg / kItemSegs] = 1;  // benign race: every writer stores 1
    }
    return total;
}

// find-first mode: the smallest start position among this warp's hits of one segment goes into the search's key word.
// Positions of one segment order as slab * 512 + lane * 16 + bit, so a 32-bit warp minimum finds the smallest.
__device__ __forceinline__ void report_first(const ScanArgs &A, const uint32_t (&hm)[4], int64_t seg_v0, int lane)
{
    uint32_t off = 0xFFFFFFFFu;
#pragma unroll
    for (int sl = 3; sl >= 0; --sl)
        if (hm[sl]) off = sl * 512 + lane * 16 + (__ffs(hm[sl]) - 1);
    off = __reduce_min_sync(0xFFFFFFFFu, off);
    if (lane == 0 && off != 0xFFFFFFFFu) {
        const unsigned long long p = (unsigned long long)(seg_v0 + off + A.pos_bias);
        atomicMax(A.first_key, ((unsigned long long)A.find_epoch << 47) | (kFindMask - (p & kFindMask)));
    }
}
// The smallest position reported so far in this search, or -1.
__device__ __forceinline__ long long first_so_far(const ScanArgs &A)
{
    const unsigned long long k = __ldcg(A.first_key);
    return (uint32_t)(k >> 47) == A.find_epoch ? (long long)(kFindMask - (k & kFindMask)) : -1ll;
}

// A warp switches to dense_tile() for its next tile when, on average, this many of its lanes held
// candidates in each segment of the current tile: then the any-pass + vote + recompute of the sparse
// path costs more than building every lane's masks right away.
// Measured (profiles/dense_lanes_r02.txt): long patterns gain from the dense path early -- its ONE verification per segment
// replaces one per slab, and a 25-byte comparison is what costs -- (m = 25 on English prose: 1.50 -> 2.03 TB/s at 3),
// short ones lose (m = 8: 2.24 -> 1.77 TB/s at 3; DNA m = 7: 1.94 -> 1.51), so the threshold follows the pattern length.
constexpr uint32_t kDenseLanesLong = 3, kDenseLanesShort = 6;

struct VerifyCtx {
    const uint8_t *vbase, *pat;
    const uint32_t *rpat;
    const int32_t *bad, *good;
    bool exact_filter, all_valid;
};

// Dense text (periodic worst cases: most lanes of the previous tile had hits): this warp's part of
// a tile without the any-pass and the vote -- every lane builds its masks right away.  Kept out of
// line so the common path of scan_kernel stays exactly the sparse filter loop.  Returns the hits
// found (count-only mode adds them up) with bit 63 set while the text is still dense.
template <Filter F, int TILE, bool POSITIONS, bool FOLD>
__device__ __forceinline__ unsigned long long dense_tile_body(const ScanArgs &A, const uint8_t *st, int64_t tile_v0,
                                                              VerifyCtx vc, int warp, int lane)
{
    constexpr int WARP_BYTES = TILE / kConsumerWarps;
    constexpr int OFFS = filter_owner_offset(F);
    unsigned long long found = 0;
    uint32_t cand_lanes = 0, tile_total = 0;
    const uint32_t tile_seg0 = (uint32_t)(tile_v0 / kSegBytes);   // 32-bit segment index of the tile's first segment
    for (int sg = 0; sg < WARP_BYTES / kSegBytes; ++sg) {
        const uint32_t seg_off = warp * WARP_BYTES + sg * kSegBytes;
        const int64_t seg_p0 = tile_v0 + seg_off + lane * 16 + OFFS;
        uint4 w[4];
        uint32_t w4[4], hm[4];
        load_segment(st + seg_off, lane, w, w4);
        // candidate masks of all four slabs, then ONE verification for the lane's whole share of the segment: candidates
        // of different slabs usually sit in different lanes, and the lanes of one call verify concurrently
        unsigned long long cand64 = 0;
#pragma unroll
        for (int sl = 0; sl < 4; ++sl) {
            uint32_t cand = filter_mask<F>(w[sl], w4[sl], A);
            if (!vc.all_valid) cand &= valid_bits(seg_p0 + sl * 512, A.vmin, A.vmax);
            cand64 |= (unsigned long long)cand << (16 * sl);
        }
        cand_lanes += __popc(__ballot_sync(0xFFFFFFFFu, cand64 != 0));
        if (cand64 && !vc.exact_filter)
            cand64 = verify_candidates<FOLD>(cand64, vc.vbase, seg_p0, A.m, vc.pat, vc.rpat, vc.bad, vc.good, A.verify_smem != 0);
#pragma unroll
        for (int sl = 0; sl < 4; ++sl) hm[sl] = (uint32_t)(cand64 >> (16 * sl)) & 0xFFFFu;
        const uint32_t seg_hits = __popcll(cand64);
        const uint32_t hit_lanes = __ballot_sync(0xFFFFFFFFu, seg_hits != 0);
        found += seg_hits;
        if (!POSITIONS && A.find_epoch && hit_lanes) report_first(A, hm, tile_v0 + seg_off + OFFS, lane);
        if (POSITIONS && hit_lanes) tile_total += publish_segment(A, tile_seg0 + seg_off / kSegBytes, hm, seg_hits, lane);
    }
    if (POSITIONS && tile_total && lane == 0)
        atomicAdd(&A.block_sum[tile_seg0 / kBlockSegs], tile_total);   // a tile lies inside one 2 MiB block
    return found | (cand_lanes >= A.dense_lanes * (WARP_BYTES / kSegBytes) ? (1ull << 63) : 0ull);
}
// Out of line for the kernels that verify (their common path must stay exactly the sparse filter loop); the m = 1 and
// m = 2 kernels, whose filter is exact and whose dense path is the one natural-language text lives in, inline the body:
// out of line the kernel arguments are reached through a generic pointer (LD.E, a long-scoreboard stall per segment:
// profiles/r02_ncu_scan_eng_is.txt), inline they are constant-bank operands ('is' on English prose count-only 4.52 ->
// 4.86 TB/s, ' ' 5.25 -> 5.78).  m = 3 stays out of line: inlined, its SPARSE path lost 7 % (bytes256: 6.6 -> 5.95 TB/s).
template <Filter F, int TILE, bool POSITIONS, bool FOLD>
__device__ __noinline__ unsigned long long dense_tile(const ScanArgs &A, const uint8_t *st, int64_t tile_v0, VerifyCtx vc, int warp, int lane)
{
    return dense_tile_body<F, TILE, POSITIONS, FOLD>(A, st, tile_v0, vc, warp, lane);
}

// FOLD: case-insensitive scan (BMX_IGNORE_CASE).  The pattern block is folded on the host; the kernel folds each
// staged tile (fold_stage) and the bytes it verifies from global memory.
template <Filter F, int TILE, bool POSITIONS, bool FOLD>
__global__ void __launch_bounds__(kThreads, 2) scan_kernel(const __grid_constant__ ScanArgs A)
{
    constexpr int WARP_BYTES = TILE / kConsumerWarps;   // contiguous bytes owned by one warp
    constexpr int OFFS = filter_owner_offset(F);        // start position of bit 0 relative to the chunk
    constexpr int SEGS = WARP_BYTES / kSegBytes;        // 2 KiB segments per warp per tile
    static_assert(SEGS >= 1 && SEGS * kSegBytes * kConsumerWarps == TILE, "tile must be a multiple of 16 KiB");
    constexpr int kSegUnroll = F == kWindow4 ? 1 : SEGS;

    extern __shared__ __align__(128) uint8_t smem[];
    SmemCtl *ctl = reinterpret_cast<SmemCtl *>(smem);
    uint8_t *stages = smem + kCtlBytes + (filter_is_set(F) ? A.multi_smem : 0u);

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const uint32_t S = A.stages;
    // multi-pattern variant: the shared candidate table sits between the control block and the stages.  A dictionary
    // keeps bitmap | occupancy bits | (table, when it is staged) there; its directory stays in global memory.
    MultiSmem M;
    M.bits = reinterpret_cast<const uint32_t *>(smem + kCtlBytes);
    if (F == kDict) {
        const size_t occ_off = (size_t)kMultiBitmapWords * 4;
        M.occ = reinterpret_cast<const uint32_t *>(smem + kCtlBytes + occ_off);
        M.table = A.mtable_smem ? reinterpret_cast<const uint2 *>(smem + kCtlBytes + occ_off + ((size_t)1 << A.mocc_log2) / 8) : A.g_mtable;
        M.dir = A.g_mdir;
    } else {
        M.occ = nullptr;
        M.table = reinterpret_cast<const uint2 *>(smem + kCtlBytes + (size_t)kMultiBitmapWords * 4);
        M.dir = reinterpret_cast<const uint2 *>(smem + kCtlBytes + (size_t)kMultiBitmapWords * 4 + (size_t)kMultiSlots * 8);
    }
    const uint8_t *mblob = (filter_is_set(F) && A.multi_blob_smem) ? reinterpret_cast<const uint8_t *>(ctl->good) : A.g_mblob;

    // Fetches one tile (plus the 16 bytes in front of it and the halo behind it) into pipeline slot s.
    auto fetch_tile = [&](uint32_t tile, uint32_t s) {
        ctl->slot_tile[s] = (int32_t)tile;
        uint8_t *dst = stages + (size_t)s * A.stage_stride;
        const int64_t v0 = (int64_t)tile * TILE;
        int64_t src_v = v0 - kPre;
        if (tile == 0) {  // nothing in front of the first tile
            src_v = 0;
            dst += kPre;
        }
        int64_t end_v = v0 + TILE + (int64_t)A.halo;
        if (end_v > A.vlen) end_v = A.vlen;
        const uint32_t bytes = (uint32_t)(end_v - src_v);
        const uint32_t bulk = bytes & ~15u;
        // ragged tail of the text (< 16 bytes, last tiles only): plain byte copies
        for (uint32_t j = bulk; j < bytes; ++j) dst[j] = A.vtext[src_v + j];
        if (bulk) {
            mbar_arrive_expect_tx(&ctl->full[s], bulk);
            tma_bulk_g2s(dst, A.vtext + src_v, bulk, &ctl->full[s]);
        } else {
            mbar_arrive(&ctl->full[s]);
        }
    };

    // The producer thread sets up the pipeline and has the CTA's first tile -- statically tile blockIdx.x, the
    // grid never exceeds the tile count -- in flight before anything else happens: the ticket round trip and
    // the staging of the tables below overlap the first HBM access instead of preceding it.
    const bool is_producer = tid == kConsumerThreads;
    uint32_t next_tile = 0;
    if (is_producer) {
        for (uint32_t s = 0; s < S; ++s) {
            mbar_init(&ctl->full[s], 1);
            mbar_init(&ctl->empty[s], kConsumerWarps);
        }
        mbar_fence_init();
        fetch_tile(blockIdx.x, 0);
        next_tile = gridDim.x + atomicAdd(A.tile_counter, 1u);  // tickets hand out the tiles behind the static ones
    }
    if (A.pat_smem) {
        for (int i = tid; i < 256; i += kThreads) ctl->bad[i] = A.g_bad[i];
        for (int i = tid; i < A.m; i += kThreads) {
            ctl->good[i] = A.g_good[i];
            ctl->pat[i] = A.g_pat[i];
        }
        for (int i = tid; i < (A.m >> 2); i += kThreads) {   // pattern words counted from the right end
            const uint8_t *q = A.g_pat + (A.m - 4 - 4 * i);
            ctl->rpat[i] = (uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24);
        }
    }
    if (F == kShiftAnd) {
        for (int i = tid; i < 256; i += kThreads) ctl->sa_mask[i] = 0u;
    }
    if (F == kMulti) {
        uint4 *dst = reinterpret_cast<uint4 *>(smem + kCtlBytes);
        const uint4 *b4 = reinterpret_cast<const uint4 *>(A.g_mbits), *t4 = reinterpret_cast<const uint4 *>(A.g_mtable),
                    *d4 = reinterpret_cast<const uint4 *>(A.g_mdir);
        constexpr int NB = kMultiBitmapWords / 4, NT = kMultiSlots / 2, ND = kMultiMaxPatterns / 2;
        for (int i = tid; i < NB; i += kThreads) dst[i] = b4[i];
        for (int i = tid; i < NT; i += kThreads) dst[NB + i] = t4[i];
        for (int i = tid; i < ND; i += kThreads) dst[NB + NT + i] = d4[i];
    }
    if (F == kDict) {   // the image puts bitmap, occupancy bits and table one behind the other, as they are staged
        uint4 *dst = reinterpret_cast<uint4 *>(smem + kCtlBytes);
        const uint4 *src = reinterpret_cast<const uint4 *>(A.g_mbits);
        const uint32_t nvec = (uint32_t)(((size_t)kMultiBitmapWords * 4 + ((size_t)1 << A.mocc_log2) / 8 +
                                          (A.mtable_smem ? ((size_t)8 << A.mslots_log2) : 0)) / 16);
        for (uint32_t i = tid; i < nvec; i += kThreads) dst[i] = src[i];
    }
    if (filter_is_set(F)) {
        if (A.multi_blob_smem) {   // the patterns themselves ride in the good-suffix area of the control block (unused here)
            uint4 *bd = reinterpret_cast<uint4 *>(ctl->good);
            const uint4 *bs = reinterpret_cast<const uint4 *>(A.g_mblob);
            for (uint32_t i = tid; i < A.multi_blob_smem / 16u; i += kThreads) bd[i] = bs[i];
        }
    }
    __syncthreads();
    if (F == kShiftAnd) {
        for (int i = tid; i < A.m; i += kThreads) atomicOr(&ctl->sa_mask[A.g_pat[i]], 1u << i);
        __syncthreads();
    }

    // ------------------------------------------------------------------ producer warp
    if (warp == kConsumerWarps) {
        if (lane != 0) return;
        // slot and phase of round `it` are it % S and (it / S) & 1, kept incrementally (S is a runtime value: the division
        // cost ~25 instructions per tile in every warp)
        uint32_t s = 1u % S, ph = (1u / S) & 1u;
        for (;; s = (s + 1u == S) ? 0u : s + 1u, ph ^= (s == 0u) ? 1u : 0u) {
            const uint32_t tile = next_tile;
            bool live = tile < A.num_tiles;
            if (!POSITIONS && A.find_epoch && live) {  // find-first: nothing at or behind a tile that starts past the best hit can win
                const long long found = first_so_far(A);
                if (found >= 0 && (long long)tile * TILE + OFFS + A.pos_bias > found) live = false;
            }
            if (live) next_tile = gridDim.x + atomicAdd(A.tile_counter, 1u);  // ticket for the next round, in flight during the wait
            mbar_wait(&ctl->empty[s], ph ^ 1u);
            if (!live) {
                ctl->slot_tile[s] = -1;
                mbar_arrive(&ctl->full[s]);
                break;
            }
            fetch_tile(tile, s);
        }
        return;
    }

    // ------------------------------------------------------------------ consumer warps
    const uint8_t *pat = A.pat_smem ? ctl->pat : A.g_pat;
    const int32_t *bad = A.pat_smem ? ctl->bad : A.g_bad;
    const int32_t *good = A.pat_smem ? ctl->good : A.g_good;
    const uint32_t *rpat = A.pat_smem ? ctl->rpat : nullptr;
    // (m decides only for the WINDOW kinds: the others pass a constant, so the call folds in the front end and the
    // out-of-line dense_tile is compiled knowing the value)
    const bool exact_filter = filter_exact(F, filter_variant(F) == BMX_VARIANT_WINDOW ? A.m : 0);
    // flagged chunks are checked by the whole warp when pattern and window both sit in shared memory (m <= kPatSmemMax)
    const bool coop = !filter_never_verifies(F) && !exact_filter && A.pat_smem != 0u && A.verify_smem != 0u && A.coop_verify != 0u;
    const uint32_t *patw = reinterpret_cast<const uint32_t *>(ctl->pat);
    CoopLane cl{};
    if (coop) cl = coop_lane_setup<OFFS>(patw, A.m, lane);
    unsigned long long my_count = 0;  // count-only mode
    bool dense_mode = false;          // per warp: candidates in most lanes -> next tile takes dense_tile()

    for (uint32_t s = 0u, ph = 0u;; s = (s + 1u == S) ? 0u : s + 1u, ph ^= (s == 0u) ? 1u : 0u) {
        mbar_wait(&ctl->full[s], ph);
        const int32_t tile_s = ctl->slot_tile[s];
        if (tile_s < 0) break;   // taken by every warp at once: each warp below reaches the fold's barrier
        if constexpr (FOLD) {
            fold_stage(stages + (size_t)s * A.stage_stride, A.stage_stride, tid);
            bar_sync_consumers();
        }
        const uint32_t tile = (uint32_t)tile_s;
        const uint8_t *st = stages + (size_t)s * A.stage_stride + kPre;  // st[0] = first byte of the tile
        const int64_t tile_v0 = (int64_t)tile * TILE;
        const uint32_t tile_seg0 = tile * (uint32_t)(TILE / kSegBytes);   // 32-bit segment index of the tile's first segment
        const uint8_t *vbase = A.verify_smem ? (st - tile_v0) : A.vtext;  // text(v) = vbase[v]
        // every start position owned by this tile may be reported (false only at the text's ends)
        const bool all_valid = tile_v0 + OFFS >= A.vmin && tile_v0 + (TILE - 1) + OFFS <= A.vmax;

        bool took_dense = false;
        if constexpr (F != kShiftAnd && !filter_is_set(F)) {
            if (dense_mode) {
                const VerifyCtx vc{vbase, pat, rpat, bad, good, exact_filter, all_valid};
                unsigned long long r;
                if constexpr (F == kBytes1 || F == kBytes2) r = dense_tile_body<F, TILE, POSITIONS, FOLD>(A, st, tile_v0, vc, warp, lane);
                else r = dense_tile<F, TILE, POSITIONS, FOLD>(A, st, tile_v0, vc, warp, lane);
                dense_mode = (r >> 63) != 0;
                if (!POSITIONS) my_count += r & ~(1ull << 63);
                took_dense = true;
            }
        }
        if (!took_dense) {
            uint32_t cand_lanes = 0, tile_total = 0;
            // (the 4-byte WINDOW kernel is ALU-bound and its two unrolled segments gave the compiler nothing to overlap: one
            // rolled copy measured +5 % on bytes256 m = 4; every other kernel is faster unrolled)
#pragma unroll(kSegUnroll)
            for (int sg = 0; sg < SEGS; ++sg) {
                uint32_t hm[4] = {0u, 0u, 0u, 0u};
                uint32_t seg_hits = 0;
                const uint32_t seg_off = warp * WARP_BYTES + sg * kSegBytes;   // this warp's 2 KiB segment
                const int64_t seg_p0 = tile_v0 + seg_off + lane * 16 + OFFS;   // start position of bit 0, slab 0
                bool has_hits = false;
                if (F == kShiftAnd) {
#pragma unroll
                    for (int sl = 0; sl < 4; ++sl) {
                        uint32_t hits = shiftand_chunk(st + seg_off + sl * 512 + lane * 16, A.m, ctl->sa_mask);
                        if (hits) hits &= valid_bits(seg_p0 + sl * 512, A.vmin, A.vmax);
                        hm[sl] = hits;
                        seg_hits += __popc(hits);
                    }
                    has_hits = __any_sync(0xFFFFFFFFu, seg_hits != 0);
                } else {
                    uint4 w[4];
                    uint32_t w4[4];
                    load_segment(st + seg_off, lane, w, w4);
                    uint32_t w5[4] = {0u, 0u, 0u, 0u};
                    if (filter_is_set(F) && A.hmul2 != 0u) load_second_after(st + seg_off, lane, w, w5);
                    bool any[4];
#pragma unroll
                    for (int sl = 0; sl < 4; ++sl)
                        any[sl] = filter_is_set(F) ? multi_any(w[sl], w4[sl], w5[sl], A.hmul, A.hmul2, M.bits) : filter_any<F>(w[sl], w4[sl], A);
                    const uint32_t vote = __ballot_sync(0xFFFFFFFFu, any[0] | any[1] | any[2] | any[3]);
                    if (vote) {  // warp-uniform and rare: the common path ends at this branch
                        if (filter_is_set(F)) {
#pragma unroll
                            for (int sl = 0; sl < 4; ++sl) {
                                if (any[sl]) {
                                    hm[sl] = multi_chunk<F>(A, M, mblob, w[sl], w4[sl], w5[sl], seg_p0 + sl * 512 - OFFS, vbase);
                                    seg_hits += __popc(hm[sl]);
                                }
                            }
                        } else if (coop) {
                            // flagged chunks one after the other, each checked by the whole warp (coop_verify16)
#pragma unroll
                            for (int sl = 0; sl < 4; ++sl) {
                                uint32_t flagged = __ballot_sync(0xFFFFFFFFu, any[sl]);
                                while (flagged) {
                                    const int src = __ffs(flagged) - 1;
                                    flagged &= flagged - 1;
                                    const int32_t rel = (int32_t)seg_off + sl * 512 + src * 16;
                                    uint32_t h16 = coop_verify16<OFFS>(st + rel, cl, patw, lane);
                                    if (!all_valid && h16) h16 &= valid_bits(tile_v0 + rel + OFFS, A.vmin, A.vmax);
                                    if (lane == src) hm[sl] = h16;
                                }
                                seg_hits += __popc(hm[sl]);
                            }
                        } else {
#pragma unroll
                            for (int sl = 0; sl < 4; ++sl) {
                                if (any[sl]) {
                                    const int64_t p0 = seg_p0 + sl * 512;
                                    uint32_t cand = filter_mask<F>(w[sl], w4[sl], A);
                                    if (!all_valid) cand &= valid_bits(p0, A.vmin, A.vmax);
                                    if (cand)
                                        hm[sl] = exact_filter ? cand : (uint32_t)verify_candidates<FOLD>(cand, vbase, p0, A.m, pat, rpat, bad, good, A.verify_smem != 0);
                                    seg_hits += __popc(hm[sl]);
                                }
                            }
                        }
                        has_hits = __any_sync(0xFFFFFFFFu, seg_hits != 0);
                        cand_lanes += __popc(vote);
                    }
                }
                if (has_hits) {
                    if (!POSITIONS) {
                        my_count += seg_hits;
                        if (A.find_epoch) report_first(A, hm, tile_v0 + seg_off + OFFS, lane);
                    } else tile_total += publish_segment(A, tile_seg0 + seg_off / kSegBytes, hm, seg_hits, lane);
                }
            }
            if (POSITIONS && tile_total && lane == 0)  // a warp's 4 KiB of a tile lie inside one 2 MiB block
                atomicAdd(&A.block_sum[tile_seg0 / kBlockSegs], tile_total);   // a tile lies inside one 2 MiB block
            dense_mode = cand_lanes >= A.dense_lanes * SEGS;  // takes effect with the next tile
        }
        // every lane is done reading the stage: hand it back to the producer
        __syncwarp();
        if (lane == 0) mbar_arrive(&ctl->empty[s]);
    }

    if (!POSITIONS) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) my_count += __shfl_xor_sync(0xFFFFFFFFu, my_count, o);
        if (lane == 0 && my_count) atomicAdd(A.scan_count, my_count);
        // the CTA that finishes last folds this scan's count into the running total of the search
        __threadfence();
        bar_sync_consumers();
        if (tid == 0 && atomicAdd(A.tile_counter + 1, 1u) == gridDim.x - 1) {
            __threadfence();
            const unsigned long long running = (A.first_scan ? 0ull : *A.count_acc) + __ldcg(A.scan_count);
            *A.count_acc = running;
            if (A.host_count) {
                A.host_count[0] = running;
                if (A.find_epoch) A.host_count[1] = (unsigned long long)first_so_far(A);
            }
            // leave the header as it was found (all zero): a count-only scan needs no memset before the next one
            A.tile_counter[0] = 0u;
            A.tile_counter[1] = 0u;
            *A.scan_count = 0ull;
        }
        return;
    }

    // ---- ordered emission, step 2 (fused): the CTA that finishes last turns the per-block hit
    // counts into exclusive bases and the running total, so the expand kernel can start right away.
    __threadfence();  // this CTA's counts, masks and block sums are visible before it reports in
    bar_sync_consumers();
    if (tid == 0) ctl->is_last = atomicAdd(A.tile_counter + 1, 1u) == gridDim.x - 1 ? 1u : 0u;
    bar_sync_consumers();
    if (!ctl->is_last) return;
    __threadfence();
    // Chunks of 2048 blocks: thread t owns 8 consecutive blocks of the chunk and loads their sums with 8
    // independent loads (one round trip -- a load-add loop here cost 2 x 8 dependent L2 round trips at the very
    // end of the kernel), the CTA scans the 256 partial sums, every thread writes its bases and dense blocks.
    constexpr uint32_t kRun = 8;
    unsigned long long hits_carry = 0;  // hits / dense blocks in front of the chunk
    uint32_t dense_carry = 0;
    for (uint32_t c0 = 0; c0 < A.num_blocks; c0 += kConsumerThreads * kRun) {
        const uint32_t b0 = c0 + (uint32_t)tid * kRun;
        uint32_t v[kRun];
#pragma unroll
        for (uint32_t j = 0; j < kRun; ++j) v[j] = b0 + j < A.num_blocks ? __ldcg(&A.block_sum[b0 + j]) : 0u;
        unsigned long long hits = 0;
        uint32_t ndense = 0;
#pragma unroll
        for (uint32_t j = 0; j < kRun; ++j) {
            hits += v[j];
            ndense += v[j] >= kDenseBlockHits ? 1u : 0u;
        }
        unsigned long long hits_incl = hits;
        uint32_t dense_incl = ndense;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long th = __shfl_up_sync(0xFFFFFFFFu, hits_incl, o);
            const uint32_t td = __shfl_up_sync(0xFFFFFFFFu, dense_incl, o);
            if (lane >= o) {
                hits_incl += th;
                dense_incl += td;
            }
        }
        if (lane == 31) {
            ctl->scan_warp[warp] = hits_incl;
            ctl->scan_dense[warp] = dense_incl;
        }
        bar_sync_consumers();
        unsigned long long hits_before = hits_carry + hits_incl - hits, chunk_hits = 0;
        uint32_t dense_before = dense_carry + dense_incl - ndense, chunk_dense = 0;
#pragma unroll
        for (int w = 0; w < kConsumerWarps; ++w) {
            const unsigned long long wh = ctl->scan_warp[w];
            const uint32_t wd = ctl->scan_dense[w];
            if (w < warp) {
                hits_before += wh;
                dense_before += wd;
            }
            chunk_hits += wh;
            chunk_dense += wd;
        }
#pragma unroll
        for (uint32_t j = 0; j < kRun; ++j) {
            if (b0 + j < A.num_blocks) {
                A.block_base[b0 + j] = hits_before;
                hits_before += v[j];
                if (v[j] >= kDenseBlockHits) A.dense_list[dense_before++] = b0 + j;  // ascending: expand_kernel walks it in ticket order
            }
        }
        hits_carry += chunk_hits;
        dense_carry += chunk_dense;
        bar_sync_consumers();  // scan_warp / scan_dense are rewritten by the next chunk
    }
    if (tid == 0) {
        const unsigned long long running = (A.first_scan ? 0ull : *A.carry_in) + hits_carry;
        *A.carry_out = running;
        if (A.host_count) *A.host_count = running;
        A.tile_counter[3] = dense_carry;
    }
}

// ---------------------------------------------------------------------------------------------
// Ordered emission, step 3: hit masks -> positions at their exact ranks (one CTA per 2 MiB block)
// ---------------------------------------------------------------------------------------------
constexpr int kExpandThreads = 256;
constexpr int kExpandWarps = kExpandThreads / 32;
constexpr uint32_t kStageThreshold = 96;  // segments with more hits go through shared memory
constexpr uint32_t kSoloMaxHits = 64;     // segments with at most this many hits are expanded by a single lane
constexpr uint32_t kFlatMaxHits = 1024;   // items (16 segments) with at most this many hits are expanded flat
constexpr int kSparseSegs = 3;            // items with at most this many segments holding hits read only those segments

// Warp-cooperative store of out[0..limit) = value(r) with 16-byte vector stores: lane l writes the
// element pairs (2l, 2l+1) + 64j of the 16-byte aligned middle part, one lane each the ragged ends.
template <typename F>
__device__ __forceinline__ void store_run(int64_t *out, uint32_t limit, int lane, F value)
{
    const uint32_t head = (uint32_t)((reinterpret_cast<uintptr_t>(out) >> 3) & 1u);  // 1: out[0] is not 16 B aligned
    if (head && lane == 0 && limit) out[0] = value(0);
    const uint32_t pairs = limit > head ? (limit - head) >> 1 : 0u;
    longlong2 *out2 = reinterpret_cast<longlong2 *>(out + head);
#pragma unroll 4
    for (uint32_t q = lane; q < pairs; q += 32) {
        const uint32_t r = head + 2 * q;
        longlong2 v;
        v.x = value(r);
        v.y = value(r + 1);
        out2[q] = v;
    }
    const uint32_t tail = head + 2 * pairs;
    if (tail < limit && lane == 31) out[tail] = value(tail);
}

// Work item = 16 segments = 32 KiB of text, expanded by ONE warp (no block-wide barriers):
//   rank of the item = carry + block base + hits of the block's segments in front of it (the warp
//   sums up to 1024 16-bit counts with 4 x LDG.128 per lane), then a 16-lane scan ranks its segments.
// Lane l of warp g probes the flag of item (32*round + l) * #warps + g, so one round of loads finds
// all work of a sparse text (every flagged item gets its own warp), and a dense text spreads evenly.
__device__ __forceinline__ void expand_segment(const ScanArgs &A, uint32_t seg, uint32_t cnt, unsigned long long seg_rank,
                                               const uint32_t (&hm)[4], uint16_t *stg, int lane)
{
    const int64_t cap = A.pos_cap;
    if ((int64_t)seg_rank >= cap) return;  // truncated output keeps the smallest positions
    const int64_t seg_pos = (int64_t)seg * kSegBytes + A.owner_offset + A.pos_bias;
    const int64_t room = cap - (int64_t)seg_rank;  // > 0 here
    const uint32_t limit = room < (int64_t)cnt ? (uint32_t)room : cnt;
    int64_t *out = A.pos_out + seg_rank;
    if (cnt == kSegBytes) {
        // every start position of the segment matches (periodic worst case, e.g. 'aaa' in
        // 'aaaa...'): ranks are affine in the position, so the warp streams them out directly
        store_run(out, limit, lane, [&](uint32_t r) { return seg_pos + (int64_t)r; });
        return;
    }
    // one warp scan for all four slabs: two words of two 16-bit counters each
    uint32_t p01 = __popc(hm[0]) | (__popc(hm[1]) << 16);
    uint32_t p23 = __popc(hm[2]) | (__popc(hm[3]) << 16);
    const uint32_t k01 = p01, k23 = p23;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t01 = __shfl_up_sync(0xFFFFFFFFu, p01, o);
        const uint32_t t23 = __shfl_up_sync(0xFFFFFFFFu, p23, o);
        if (lane >= o) {
            p01 += t01;
            p23 += t23;
        }
    }
    const uint32_t tot01 = __shfl_sync(0xFFFFFFFFu, p01, 31), tot23 = __shfl_sync(0xFFFFFFFFu, p23, 31);
    const uint32_t e01 = p01 - k01, e23 = p23 - k23;  // exclusive prefixes inside each slab
    uint32_t start[4];
    start[0] = e01 & 0xFFFFu;
    start[1] = (tot01 & 0xFFFFu) + (e01 >> 16);
    start[2] = (tot01 & 0xFFFFu) + (tot01 >> 16) + (e23 & 0xFFFFu);
    start[3] = (tot01 & 0xFFFFu) + (tot01 >> 16) + (tot23 & 0xFFFFu) + (e23 >> 16);
    if (cnt >= kStageThreshold) {
        // dense segment: scatter 16-bit local offsets into shared memory (XOR-swizzled so the
        // 16 consecutive ranks of a lane do not pile up on 4 banks), then write coalesced
#pragma unroll
        for (int sl = 0; sl < 4; ++sl) {
            uint32_t r = start[sl];
            const uint32_t local0 = sl * 512 + lane * 16;
            uint32_t h = hm[sl];
            while (h) {
                const uint32_t bit = __ffs(h) - 1;
                h &= h - 1;
                stg[r ^ ((r >> 4) & 15u)] = (uint16_t)(local0 + bit);
                ++r;
            }
        }
        __syncwarp();
        store_run(out, limit, lane, [&](uint32_t r) { return seg_pos + (int64_t)stg[r ^ ((r >> 4) & 15u)]; });
        __syncwarp();
    } else {
#pragma unroll
        for (int sl = 0; sl < 4; ++sl) {
            uint32_t r = start[sl];
            const uint32_t local0 = sl * 512 + lane * 16;
            uint32_t h = hm[sl];
            while (h) {
                const uint32_t bit = __ffs(h) - 1;
                h &= h - 1;
                if (r < limit) out[r] = seg_pos + local0 + bit;
                ++r;
            }
        }
    }
}

// `share`/`member`: the item's segments are dealt round-robin to `share` cooperating warps.
__device__ __forceinline__ void expand_item(const ScanArgs &A, uint32_t item, unsigned long long carry, uint16_t *stg, int lane,
                                            uint32_t share, uint32_t member)
{
    const uint32_t blk = item / kExpandSplit;
    const uint32_t first = (item % kExpandSplit) * kItemSegs;  // first segment of the item inside its block
    // hits of the block's segments in front of this item: lane l covers counts [32l, 32l+32)
    const uint32_t blk_seg0 = blk * kBlockSegs;
    uint32_t acc = 0;
    if ((uint32_t)lane * 32u < first) {
        const uint4 *cp = reinterpret_cast<const uint4 *>(A.seg_count + blk_seg0 + lane * 32);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint4 v = cp[q];  // 8 counts; pairs share a word and stay below 2^16 when summed 16 at a time
            const uint32_t ws[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if ((uint32_t)lane * 32u + q * 8u + j * 2u < first) acc += ws[j];
        }
    }
    uint32_t before = (acc & 0xFFFFu) + (acc >> 16);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xFFFFFFFFu, before, o);

    const uint32_t seg0 = blk_seg0 + first;
    const uint32_t c = (lane < kItemSegs && seg0 + lane < A.num_segs) ? A.seg_count[seg0 + lane] : 0u;
    uint32_t incl = c;
#pragma unroll
    for (int o = 1; o < kItemSegs; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += t;
    }
    const unsigned long long item_rank = carry + A.block_base[blk] + before;
    // Items with moderately many hits (natural-language text: a dozen hits per 2 KiB segment) are expanded
    // "flat": lane l takes the 64 consecutive masks l*64 .. l*64+63 of the item (8 x LDG.128 issued together),
    // one warp scan over the lanes' popcounts ranks every lane inside the item, and each lane stores its own
    // hits.  No per-segment scans, all 32 lanes busy: a fifth of the instructions of the paths below.
    const uint32_t item_total = __shfl_sync(0xFFFFFFFFu, incl, kItemSegs - 1);
    // Sparse items (the usual case of a sparse text: one or two of the 16 segments hold a hit or a few): only those
    // segments are read -- lane l takes the 64 start positions 64 l .. 64 l + 63 of the segment as ONE 8-byte load, a
    // warp scan ranks the lanes, every lane stores its own hits.  ~70 warp-instructions per such segment where the flat
    // path below spends ~400 on the item (profiles/r02_ncu_expand_dna8.txt: 425 instructions per hit on DNA, m = 8).
    const uint32_t seg_vote = __ballot_sync(0xFFFFFFFFu, c != 0u);
    if (share == 1 && __popc(seg_vote) <= kSparseSegs && item_total <= kStageThreshold) {   // (few hits: no full segments either)
        for (uint32_t v = seg_vote; v; v &= v - 1) {
            const int src = __ffs(v) - 1;
            const uint32_t seg = seg0 + (uint32_t)src;
            const unsigned long long seg_rank = item_rank + __shfl_sync(0xFFFFFFFFu, incl - c, src);
            const uint2 mk = reinterpret_cast<const uint2 *>(A.mask16 + (size_t)seg * kSegChunks)[lane];
            const uint32_t mine = __popc(mk.x) + __popc(mk.y);
            uint32_t upto = mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, upto, o);
                if (lane >= o) upto += t;
            }
            const unsigned long long rank = seg_rank + (upto - mine);
            const int64_t room = A.pos_cap - (int64_t)rank;   // truncated output keeps the smallest positions
            if (mine != 0u && room > 0) {
                int64_t *out = A.pos_out + rank;
                const int64_t pos0 = (int64_t)seg * kSegBytes + A.owner_offset + A.pos_bias + lane * 64;
                uint32_t written = 0;
                for (uint32_t w = mk.x; w; w &= w - 1, ++written)
                    if ((int64_t)written < room) out[written] = pos0 + (__ffs(w) - 1);
                for (uint32_t w = mk.y; w; w &= w - 1, ++written)
                    if ((int64_t)written < room) out[written] = pos0 + 32 + (__ffs(w) - 1);
            }
        }
        return;
    }
    if (share == 1 && item_total <= kFlatMaxHits) {
        const uint32_t cs = __shfl_sync(0xFFFFFFFFu, c, lane >> 1);   // hits of the segment this lane's masks belong to
        uint4 v[8];
        const uint4 *mp = reinterpret_cast<const uint4 *>(A.mask16 + (size_t)seg0 * kSegChunks) + lane * 8;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            // segments without hits never wrote their masks; full segments did not need to
            v[u] = cs == 0 ? make_uint4(0u, 0u, 0u, 0u)
                           : (cs == kSegBytes ? make_uint4(~0u, ~0u, ~0u, ~0u) : mp[u]);
        }
        uint32_t mine = 0;
#pragma unroll
        for (int u = 0; u < 8; ++u) mine += __popc(v[u].x) + __popc(v[u].y) + __popc(v[u].z) + __popc(v[u].w);
        uint32_t before_me = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, before_me, o);
            if (lane >= o) before_me += t;
        }
        before_me -= mine;
        const unsigned long long rank = item_rank + before_me;
        const int64_t room = A.pos_cap - (int64_t)rank;
        if (mine != 0 && room > 0) {
            // One loop per lane over its HITS: the warp runs max over lanes of `mine` iterations.  Walking the 32 words
            // of a lane in an unrolled loop with a hit loop inside each (the first version) made the warp pay every
            // word's worst lane: 1600 instructions per item on English prose (profiles/r02_ncu_expand_eng_is.txt).  The
            // lane parks its words in shared memory ([word][lane]: its own bank, whatever word each lane is at) and
            // keeps a bitmap of the nonzero ones, so "next word" is FFS + one LDS and empty words cost nothing.
            int64_t *out = A.pos_out + rank;
            const int64_t pos0 = (int64_t)seg0 * kSegBytes + A.owner_offset + A.pos_bias + lane * 1024;
            uint32_t *park = reinterpret_cast<uint32_t *>(stg) + lane;
            uint32_t nz = 0u;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const uint32_t ws[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    park[(u * 4 + k) * 32] = ws[k];
                    nz |= ws[k] ? 1u << (u * 4 + k) : 0u;
                }
            }
            uint32_t j = 0, w = 0u, written = 0;
            for (uint32_t left = mine; left; --left) {
                if (w == 0u) {   // the parked word behind bit j of nz is nonzero: one reload always suffices
                    j = __ffs(nz) - 1;
                    nz &= nz - 1;
                    w = park[j * 32];
                }
                const uint32_t b = __ffs(w) - 1;
                w &= w - 1;
                if ((int64_t)written < room) out[written] = pos0 + j * 32 + b;
                ++written;
            }
        }
        return;
    }

    // Segments with few hits are expanded by ONE lane each -- lane l walks the 128 masks of segment l,
    // 16 lanes in parallel.
    const bool solo = share == 1 && c != 0 && c <= kSoloMaxHits;
    if (solo) {
        const uint32_t seg = seg0 + lane;
        const unsigned long long seg_rank = item_rank + (incl - c);
        const int64_t room = A.pos_cap - (int64_t)seg_rank;
        if (room > 0) {
            const int64_t seg_pos = (int64_t)seg * kSegBytes + A.owner_offset + A.pos_bias;
            int64_t *out = A.pos_out + seg_rank;
            const uint4 *mp = reinterpret_cast<const uint4 *>(A.mask16 + (size_t)seg * kSegChunks);
            uint32_t written = 0;
            for (int q0 = 0; q0 < kSegChunks / 8; q0 += 8) {
                uint4 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = mp[q0 + u];  // 8 x 8 masks in flight
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const uint32_t ws[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        uint32_t w = ws[j];  // masks of chunks 8q+2j (low half) and 8q+2j+1 (high half)
                        const uint32_t local0 = ((q0 + u) * 8 + j * 2) * 16;
                        while (w) {
                            const uint32_t b = __ffs(w) - 1;
                            w &= w - 1;
                            if ((int64_t)written < room) out[written] = seg_pos + local0 + b;
                            ++written;
                        }
                    }
                }
            }
        }
    }
    uint32_t vote = __ballot_sync(0xFFFFFFFFu, c != 0 && !solo && (uint32_t)lane % share == member);
    while (vote) {
        // up to 4 segments per round: all their mask loads are issued before any is expanded
        int src[4];
        uint32_t hm[4][4];
        int k = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            src[j] = 0;
            if (vote) {
                src[j] = __ffs(vote) - 1;
                vote &= vote - 1;
                k = j + 1;
                const uint16_t *mk = A.mask16 + (size_t)(seg0 + src[j]) * kSegChunks + lane;
                const bool full = __shfl_sync(0xFFFFFFFFu, c, src[j]) == kSegBytes;  // full segments have no masks
#pragma unroll
                for (int sl = 0; sl < 4; ++sl) hm[j][sl] = full ? 0xFFFFu : mk[sl * 32];
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j < k) {
                const uint32_t cnt = __shfl_sync(0xFFFFFFFFu, c, src[j]);
                const uint32_t off = __shfl_sync(0xFFFFFFFFu, incl - c, src[j]);
                expand_segment(A, seg0 + src[j], cnt, item_rank + off, hm[j], stg, lane);
            }
        }
    }
}

__global__ void __launch_bounds__(kExpandThreads) expand_kernel(const __grid_constant__ ScanArgs A)
{
    __shared__ uint16_t s_stage[kExpandWarps][kSegBytes];
    __shared__ uint32_t s_ticket;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // Housekeeping for the NEXT scan: clear the zero-initialised scratch half that the previous scan dirtied
    // (its expand kernel has finished: stream order).  Fire-and-forget stores under this kernel's load latency,
    // instead of a memset operation in front of every scan.
    for (uint32_t i = blockIdx.x * kExpandThreads + threadIdx.x; i < A.zero_vec16; i += gridDim.x * kExpandThreads)
        static_cast<uint4 *>(A.zero_ptr)[i] = make_uint4(0u, 0u, 0u, 0u);
    const unsigned long long carry = A.first_scan ? 0ull : *A.carry_in;
    const uint32_t dense_items = A.tile_counter[3] * kExpandSplit;  // loaded up front, used by phase 2

    // ---- phase 1: items of sparse blocks, one warp per item.  Lane l of warp g probes unit l * #warps + g,
    // where a unit is one item flag if a single round of loads then covers the text, else the flags of 4
    // consecutive items (one 32-bit load: one round covers ~14 GiB with a single resident wave of CTAs).
    // A sparse text gives every flagged item its own warp, and a dense text spreads evenly.
    {
        const uint32_t gw = blockIdx.x * kExpandWarps + warp, nw = gridDim.x * kExpandWarps;
        const uint32_t items = A.num_blocks * kExpandSplit;
        const bool wide = items > nw * 32u;
        const uint32_t units = wide ? items / 4u : items, per_block = wide ? kExpandSplit / 4u : kExpandSplit;
        const uint32_t *flag4 = reinterpret_cast<const uint32_t *>(A.item_flag);
        for (uint32_t base = 0; base < units; base += nw * 32u) {
            const uint32_t mine = base + (uint32_t)lane * nw + gw;
            // both loads are issued together (no short circuit): one round trip instead of two
            uint32_t flags = mine < units ? (wide ? flag4[mine] : (uint32_t)A.item_flag[mine]) : 0u;
            const uint32_t bsum = mine < units ? A.block_sum[mine / per_block] : 0u;
            if (bsum >= kDenseBlockHits) flags = 0u;   // dense blocks belong to phase 2
#pragma unroll 1   // (unrolled, the four copies of expand_item made a 21 000-instruction kernel: cold instruction fetches sit in every call's latency chain)
            for (uint32_t k = 0; k < 4; ++k) {
                uint32_t vote = __ballot_sync(0xFFFFFFFFu, ((flags >> (8 * k)) & 0xFFu) != 0u);
                while (vote) {
                    const int src = __ffs(vote) - 1;
                    vote &= vote - 1;
                    const uint32_t unit = __shfl_sync(0xFFFFFFFFu, mine, src);
                    expand_item(A, wide ? unit * 4u + k : unit, carry, s_stage[warp], lane, 1u, 0u);
                }
            }
        }
    }

    // ---- phase 2: items of dense blocks in ticket order, a whole CTA per item (each warp two of its
    // segments).  In-order tickets keep the write frontier of the grid narrow and moving linearly, which
    // is what reaches the HBM write peak (7.2-7.6 TB/s vs 5.6-6.3 TB/s for static striding).
    if (dense_items == 0) return;
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_ticket = atomicAdd(A.tile_counter + 2, 1u);
        __syncthreads();
        const uint32_t t = s_ticket;
        if (t >= dense_items) break;
        const uint32_t item = A.dense_list[t / kExpandSplit] * kExpandSplit + t % kExpandSplit;
        if (A.item_flag[item] != 0) expand_item(A, item, carry, s_stage[warp], lane, kExpandWarps, (uint32_t)warp);
    }
}

// ---------------------------------------------------------------------------------------------
// Small utility kernels
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t mix64(uint64_t z)
{
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

struct SynthAlphabet {
    unsigned char a[256];
};

// One thread per 8-byte draw; same definition as oracle_synth_fill (oracle/bm_oracle.c).
__global__ void synth_fill_kernel(uint8_t *dst, int64_t offset, int64_t len, uint64_t seed,
                                  const __grid_constant__ SynthAlphabet alpha, int32_t sigma)
{
    const int64_t first_word = offset >> 3;
    const int64_t nwords = ((offset + len + 7) >> 3) - first_word;
    for (int64_t w = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; w < nwords; w += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t j = (uint64_t)(first_word + w);
        const uint64_t z = mix64(seed + (j + 1) * 0x9E3779B97F4A7C15ull);
        uint64_t packed = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint32_t b = (uint32_t)(z >> (8 * k)) & 0xFFu;
            packed |= (uint64_t)alpha.a[(b * (uint32_t)sigma) >> 8] << (8 * k);
        }
        const int64_t d0 = (int64_t)(j << 3) - offset;  // destination index of byte 0 of this draw
        if (d0 >= 0 && d0 + 8 <= len && ((reinterpret_cast<uintptr_t>(dst) + (uintptr_t)d0) & 7u) == 0) {
            *reinterpret_cast<uint64_t *>(dst + d0) = packed;
        } else {
            for (int k = 0; k < 8; ++k) {
                const int64_t d = d0 + k;
                if (d >= 0 && d < len) dst[d] = (uint8_t)(packed >> (8 * k));
            }
        }
    }
}

__global__ void export_result_kernel(const unsigned long long *count, const int64_t *pos, int64_t pos_cap, int64_t *dst,
                                     int64_t head)
{
    const int64_t c = (int64_t)*count;
    const int64_t held = c < pos_cap ? c : pos_cap;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        dst[0] = c;
        dst[1] = held;
    }
    const int64_t n = head < held ? head : held;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) dst[2 + i] = pos[i];
}

// ---------------------------------------------------------------------------------------------
// Host: filter choice, planning, launch
// ---------------------------------------------------------------------------------------------
Filter choose_filter(int requested_variant, const unsigned char *pat, int32_t m)
{
    // AUTO, and QGRAM for m < 7: thresholds from the measured table in DESIGN.md (profiles/variants_r01.json)
    int variant = m >= 7 ? BMX_VARIANT_QGRAM : BMX_VARIANT_WINDOW;
    if (requested_variant == BMX_VARIANT_WINDOW) variant = BMX_VARIANT_WINDOW;
    if (requested_variant == BMX_VARIANT_SHIFTAND) variant = m <= 32 ? BMX_VARIANT_SHIFTAND : BMX_VARIANT_QGRAM;
    if (variant == BMX_VARIANT_SHIFTAND) return kShiftAnd;
    // The text's alphabet is unknown here; the distinct bytes among the pattern's first 16 are the proxy.
    bool seen[256] = {false};
    int distinct = 0;
    for (int i = 0; i < m && i < 16; ++i)
        if (!seen[pat[i]]) { seen[pat[i]] = true; ++distinct; }
    if (variant == BMX_VARIANT_QGRAM) {
        // Per-residue lengths cost 3 more IMADs per word: measured -6 % on large alphabets, where the
        // shortest length is selective enough anyway, and +35 % / +32 % / +11 % on 4-letter text at m = 7 / 8 /
        // 9 (profiles/short_qgram_r01.txt).
        const int knob = env_int("BMX_QGRAM_UNIFORM", -1);   // measurement knob: 1 / 0 force one / four lengths
        const bool per_residue = knob >= 0 ? knob == 0 : (m <= 9 && distinct <= 4);
        return per_residue && m <= 10 ? kQgramPerResidue : kQgram;   // from m = 11 on every residue sees 8 bytes
    }
    if (m <= 3) return m == 1 ? kBytes1 : (m == 2 ? kBytes2 : kBytes3);
    // m = 5, 6: the 4-byte window passes 1 in 256 positions of a 4-letter text and the scan becomes
    // verification-bound (DNA: 2.0 / 2.2 TB/s).  The byte-parallel construction of the m <= 3 kernels, extended to five
    // bytes (11 instructions per word instead of 7, exact for m = 5), is chosen when the pattern has <= 4 distinct
    // bytes -- the same proxy as in the q-gram layout choice.  BMX_WINDOW5=0/1 forces either.
    if ((m == 5 || m == 6) && env_int("BMX_WINDOW5", distinct <= 4 ? 1 : 0) != 0) return kBytes5;
    return kWindow4;
}

void fill_filter_constants(Filter filter, const unsigned char *pat, int32_t m, ScanArgs *a)
{
    a->f[0] = a->f[1] = a->f[2] = a->f[3] = 0;
    a->hmul = kHashMul;
    if (filter_variant(filter) == BMX_VARIANT_QGRAM) {
        // residue r (pattern byte r on a word boundary) can use min(8, m - r) pattern bytes
        for (int r = 0; r < 4; ++r) {
            const int q2 = std::min(m - r, 8) - 4;   // bytes taken from the second word
            a->hmulr[r] = gram_multiplier(kHashMul, q2);
            a->f[r] = le_word(pat + r, 4) + a->hmulr[r] * le_word(pat + r + 4, q2);
        }
        a->hmul = a->hmulr[3];
        if (filter == kQgram) {   // one length, m - 3 bytes (at most 8), for every residue
            for (int r = 0; r < 4; ++r) {
                a->hmulr[r] = a->hmul;
                a->f[r] = le_word(pat + r, 4) + a->hmul * le_word(pat + r + 4, std::min(m - 3, 8) - 4);
            }
        }
    } else if (filter_variant(filter) == BMX_VARIANT_WINDOW) {
        for (int k = 0; k < 5; ++k) a->bcast[k] = (uint32_t)pat[std::min(k, m - 1)] * 0x01010101u;
        const int q = std::min(m, 4);
        a->f[0] = le_word(pat, q) * (q >= 4 ? 1u : (1u << (32 - 8 * q)));   // 2^(32-8q) drops the bytes beyond q
    }
}

// The scan_kernel instances of one filter kind: [case-folding][tile is 32 KiB][positions mode].  The multi-pattern kind
// has no folding instances (nullptr).
struct KernelRow {
    const void *k[2][2][2];
};
template <Filter F, bool FOLD>
static void fill_row(const void *(&k)[2][2])
{
    k[0][0] = (const void *)&scan_kernel<F, 16384, false, FOLD>;
    k[0][1] = (const void *)&scan_kernel<F, 16384, true, FOLD>;
    k[1][0] = (const void *)&scan_kernel<F, 32768, false, FOLD>;
    k[1][1] = (const void *)&scan_kernel<F, 32768, true, FOLD>;
}
template <Filter F>
static KernelRow kernels_of()
{
    KernelRow r{};
    fill_row<F, false>(r.k[0]);
    if constexpr (!filter_is_set(F)) fill_row<F, true>(r.k[1]);
    return r;
}
static const void *scan_kernel_for(Filter filter, int tile, bool positions, bool fold)
{
    static const KernelRow rows[] = {kernels_of<kQgramPerResidue>(), kernels_of<kQgram>(), kernels_of<kWindow4>(),
                                     kernels_of<kBytes1>(),          kernels_of<kBytes2>(), kernels_of<kBytes3>(),
                                     kernels_of<kBytes5>(),          kernels_of<kShiftAnd>(), kernels_of<kMulti>(),
                                     kernels_of<kDict>()};
    static_assert(sizeof rows / sizeof rows[0] == kFilterCount, "one row per filter kind, in the order of enum Filter");
    return rows[filter].k[fold][tile == 32768][positions];
}

// Device attributes (and the expand kernel's occupancy) are queried once per device, under a mutex: a search on
// a 500 KB text is launch-latency bound, and the entry points may be called from one host thread per GPU.
static std::mutex dev_mutex;

static int device_info(int device, int *sm_count, int *smem_optin, int *smem_sm, int *expand_per_sm)
{
    struct DevInfo {
        int sm_count = 0, smem_optin = 0, smem_sm = 0, expand_per_sm = 0;
    };
    static DevInfo dev_info[64];
    std::lock_guard<std::mutex> lock(dev_mutex);
    DevInfo &di = dev_info[device & 63];
    if (di.sm_count == 0) {
        DevInfo q;
        if (cudaDeviceGetAttribute(&q.sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess ||
            cudaDeviceGetAttribute(&q.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device) != cudaSuccess ||
            cudaDeviceGetAttribute(&q.smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, device) != cudaSuccess)
            return fail(BMX_E_CUDA, "cudaDeviceGetAttribute: %s", cudaGetErrorString(cudaGetLastError()));
        ScopedDevice keep;   // the occupancy query reads the current device
        cudaSetDevice(device);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&q.expand_per_sm, expand_kernel, kExpandThreads, 0) != cudaSuccess || q.expand_per_sm < 1) {
            (void)cudaGetLastError();
            q.expand_per_sm = 2;
        }
        di = q;
    }
    if (sm_count) *sm_count = di.sm_count;
    if (smem_optin) *smem_optin = di.smem_optin;
    if (smem_sm) *smem_sm = di.smem_sm;
    if (expand_per_sm) *expand_per_sm = di.expand_per_sm;
    return BMX_OK;
}

int plan_scan(int device, Filter filter, bool fold, int32_t m, bool positions, ScanArgs *a, ScanLaunch *out)
{
    int sm_count = 0, smem_optin = 0, smem_sm = 0;
    if (int rc = device_info(device, &sm_count, &smem_optin, &smem_sm, nullptr)) return rc;

    const bool multi = filter_is_set(filter);
    // profiles/tune_knobs.py: 32 KiB tiles, 2 CTAs/SM, 3 stages.  The multi-pattern variant keeps 37 KiB of tables in
    // shared memory: 16 KiB tiles leave room for a 4-stage ring next to them.
    int tile = multi ? env_int("BMX_MULTI_TILE", 16384) : env_int("BMX_TILE", 32768);
    if (tile != 16384 && tile != 32768) tile = multi ? 16384 : 32768;
    a->multi_smem = filter == kMulti  ? (uint32_t)((kMultiSmemBytes + 127) & ~size_t(127))
                    : filter == kDict ? (uint32_t)dict_smem_bytes(a->mslots_log2, a->mtable_smem, a->mocc_log2)
                                      : 0u;
    const int ctas_per_sm = std::max(1, std::min(2, env_int("BMX_CTAS_PER_SM", 2)));

    // Halo: enough for the filter's look-ahead (one more word; Shift-And reads 16+m-1 bytes per
    // chunk) and, when it fits, for verifying a whole pattern from shared memory.
    a->verify_smem = m <= kHaloSmemMax ? 1u : 0u;
    a->halo = a->verify_smem ? (uint32_t)((m + 15 + 15) & ~15) : 32u;
    a->pat_smem = (!multi && m <= kPatSmemMax) ? 1u : 0u;

    // 1 KiB per resident CTA is reserved by the driver.
    const size_t budget = std::min<size_t>((size_t)smem_optin, (size_t)smem_sm / ctas_per_sm - 1024);
    auto stages_for = [&](int t) {
        a->stage_stride = (uint32_t)((kPre + t + (int)a->halo + 127) & ~127);
        return (int)((budget - kCtlBytes - a->multi_smem) / a->stage_stride);
    };
    int stages = stages_for(tile);
    // A 32 KiB tile next to the multi-pattern table and a halo for patterns of up to 4096 bytes leaves room for one
    // stage only: such a set is scanned in 16 KiB tiles instead of failing.
    if (stages < 2 && tile == 32768) stages = stages_for(tile = 16384);
    stages = std::min(stages, std::min(kMaxStages, env_int("BMX_STAGES", kMaxStages)));
    if (stages < 2) return fail(BMX_E_NOMEM, "pattern of %d bytes leaves room for %d pipeline stages", m, stages);
    a->stages = (uint32_t)stages;

    out->filter = filter;
    out->fold = fold;
    out->tile_bytes = tile;
    out->smem_bytes = kCtlBytes + a->multi_smem + (size_t)stages * a->stage_stride;
    const int64_t tiles = (a->vlen + tile - 1) / tile;
    a->num_tiles = (uint32_t)tiles;
    a->num_segs = (uint32_t)(tiles * (tile / kSegBytes));
    a->num_blocks = (a->num_segs + kBlockSegs - 1) / kBlockSegs;
    a->owner_offset = filter_owner_offset(filter);
    a->coop_verify = env_int("BMX_COOP_VERIFY", 1) != 0 ? 1u : 0u;   // measurement knob
    // Patterns whose flagged chunks are checked by the whole warp never gain from the dense path (profiles/verify_ab_r02.txt:
    // equal or faster at every density measured): 33 lanes = never.
    const bool coop = !filter_exact(filter, m) && a->coop_verify && a->pat_smem && a->verify_smem;
    a->dense_lanes = (uint32_t)std::max(1, std::min(33, env_int("BMX_DENSE_LANES", coop ? 33 : (int)(m >= 16 ? kDenseLanesLong : kDenseLanesShort))));
    // BMX_SPARE_SMS leaves SMs free for concurrently running kernels (the NCCL collectives of a
    // multi-GPU pipeline cannot start while a persistent grid holds every SM)
    const int spare = std::max(0, std::min(sm_count - 1, env_int("BMX_SPARE_SMS", 0)));
    out->grid = (int)std::min<int64_t>(tiles, (int64_t)(sm_count - spare) * ctas_per_sm);

    const void *k = scan_kernel_for(filter, tile, positions, fold);
    {
        // the opt-in shared-memory limit of a kernel is raised once per (device, kernel, size)
        static std::map<std::pair<int, const void *>, size_t> granted;
        std::lock_guard<std::mutex> lock(dev_mutex);
        size_t &have = granted[std::make_pair(device, k)];
        if (have < out->smem_bytes) {
            if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)out->smem_bytes) != cudaSuccess)
                return fail(BMX_E_CUDA, "cudaFuncSetAttribute(smem=%zu): %s", out->smem_bytes,
                            cudaGetErrorString(cudaGetLastError()));
            have = out->smem_bytes;
        }
    }
    return BMX_OK;
}

int launch_scan(const ScanArgs &a, const ScanLaunch &l, bool positions, void *stream)
{
    const void *k = scan_kernel_for(l.filter, l.tile_bytes, positions, l.fold);
    void *params[] = {const_cast<ScanArgs *>(&a)};
    const cudaError_t e = cudaLaunchKernel(k, dim3((unsigned)l.grid), dim3(kThreads), params, l.smem_bytes,
                                           static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(BMX_E_CUDA, "scan kernel launch: %s", cudaGetErrorString(e));
    return BMX_OK;
}

int launch_emit(const ScanArgs &a, void *stream)
{
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int dev = 0, sms = 0, per_sm = 0;
    cudaGetDevice(&dev);
    if (int rc = device_info(dev, &sms, nullptr, nullptr, &per_sm)) return rc;
    // one resident wave of CTAs (a second wave would repeat the whole load-latency chain)
    const uint32_t items = a.num_blocks * kExpandSplit;
    uint32_t grid = std::min<uint32_t>((items + kExpandWarps - 1) / kExpandWarps, (uint32_t)(sms * per_sm));
    grid = std::max<uint32_t>(1u, std::min<uint32_t>(grid, (uint32_t)env_int("BMX_EXPAND_GRID", 1 << 30)));  // test knob
    expand_kernel<<<grid, kExpandThreads, 0, st>>>(a);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(BMX_E_CUDA, "expand launch: %s", cudaGetErrorString(e));
    return BMX_OK;
}

int launch_export_result(const unsigned long long *d_count, const int64_t *d_pos, int64_t pos_cap, void *d_dst, int64_t head,
                         void *stream)
{
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((head + 255) / 256, 64));
    export_result_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_count, d_pos, pos_cap,
                                                                              static_cast<int64_t *>(d_dst), head);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(BMX_E_CUDA, "export_result launch: %s", cudaGetErrorString(e));
    return BMX_OK;
}

int launch_synth_fill(void *d_text, int64_t offset, int64_t len, uint64_t seed, const unsigned char *alphabet,
                      int32_t sigma, void *stream)
{
    if (len <= 0) return BMX_OK;
    SynthAlphabet alpha;
    memset(&alpha, 0, sizeof alpha);
    memcpy(alpha.a, alphabet, (size_t)sigma);
    const int64_t nwords = ((offset + len + 7) >> 3) - (offset >> 3);
    const int block = 256;
    const int grid = (int)std::min<int64_t>((nwords + block - 1) / block, 148 * 32);
    synth_fill_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<uint8_t *>(d_text), offset,
                                                                             len, seed, alpha, sigma);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(BMX_E_CUDA, "synth_fill launch: %s", cudaGetErrorString(e));
    return BMX_OK;
}

}  // namespace bmx
