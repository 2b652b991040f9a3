// bmx_internal.h -- declarations shared by the translation units of libbmx.so (not installed).
#pragma once

#include <cstddef>
#include <cstdint>
#include <cstdlib>

#include <vector_types.h>   // uint2 (CUDA toolkit header, plain C++)

#include "../../include/bmx.h"

namespace bmx {

// ---- bmx_tables.cpp -----------------------------------------------------------------------
void build_bad_table(const unsigned char *pat, int32_t m, int32_t bad[256]);
void build_good_table(const unsigned char *pat, int32_t m, int32_t *good /* m ints */);

// ---- error plumbing (bmx_abi.cu) ----------------------------------------------------------
int fail(int code, const char *fmt, ...);

// ---- geometry of the scan kernels (bmx_scan.cu) -------------------------------------------
constexpr int kConsumerWarps = 8;                       // warps that filter/verify/emit
constexpr int kConsumerThreads = kConsumerWarps * 32;   // 256
constexpr int kThreads = kConsumerThreads + 32;         // + one producer warp (TMA issue)
constexpr int kMaxStages = 8;
constexpr int kPre = 16;            // bytes staged in front of a tile (q-gram owner offset -3)
constexpr int kPatSmemMax = 1024;   // patterns up to this length keep pattern+tables in smem
constexpr int kHaloSmemMax = 4096;  // longer patterns verify their tail from global memory

// Ordered emission works on fixed units of the (16-byte aligned) text:
//   chunk   = 16 start positions  -> one 16-bit hit mask            (mask16[v / 16])
//   segment = 128 chunks = 2 KiB  -> one 16-bit hit count           (seg_count[v / 2048])
//   block   = 1024 segments = 2 MiB -> one 32-bit hit count + base  (block_sum / block_base)
constexpr int kSegBytes = 2048;
constexpr int kSegChunks = kSegBytes / 16;   // 128
constexpr int kBlockSegs = 1024;
constexpr int64_t kBlockBytes = (int64_t)kSegBytes * kBlockSegs;   // 2 MiB

// A block is "dense" from this many hits on (6 % of its start positions): its items are then expanded in
// ticket order by whole CTAs, which keeps the write frontier narrow (profiles/micro/write_patterns.cu).
constexpr uint32_t kDenseBlockHits = 1u << 17;
constexpr int kExpandSplit = 64;                      // expand work items per block
constexpr int kItemSegs = kBlockSegs / kExpandSplit;  // 16 segments = 32 KiB of text, one warp each

// The scan kernel's filter kinds: one scan_kernel family each.  choose_filter() (bmx_scan.cu) picks one per pattern;
// the kernel, its constants and its launch plan all follow from that one value.
enum Filter : int {
    kQgramPerResidue,   // QGRAM, 7 <= m <= 10: one hash multiplier per residue (m <= 9 on small alphabets unless forced)
    kQgram,             // QGRAM: one hash multiplier for all four residues
    kWindow4,           // WINDOW, m >= 4: the 4-byte window at every position against P[0..4)
    kBytes1,            // WINDOW, m = 1, 2, 3: all m bytes at four start positions per word at once
    kBytes2,
    kBytes3,
    kBytes5,            // WINDOW, m = 5, 6 on small alphabets: the first five bytes, four start positions per word
    kShiftAnd,          // SHIFTAND, m <= 32
    kMulti,             // a multi-pattern set (bmx_multipat.cu)
    kDict,              // a dictionary (bmx_dict.cu): kMulti's filter with the table geometry set per dictionary
    kFilterCount
};

// Kinds that scan for a pattern set through the shared candidate table.
constexpr __host__ __device__ bool filter_is_set(Filter f) { return f == kMulti || f == kDict; }
// The public bmx_variant a kind belongs to (the set kinds belong to none: AUTO).
constexpr __host__ __device__ int filter_variant(Filter f)
{
    if (f == kQgramPerResidue || f == kQgram) return BMX_VARIANT_QGRAM;
    if (f == kWindow4 || f == kBytes1 || f == kBytes2 || f == kBytes3 || f == kBytes5) return BMX_VARIANT_WINDOW;
    return f == kShiftAnd ? BMX_VARIANT_SHIFTAND : BMX_VARIANT_AUTO;
}
// Start position of mask bit 0 relative to its 16-byte chunk: the q-gram hashes flag starts up to 3 bytes in front.
constexpr __host__ __device__ int filter_owner_offset(Filter f) { return f == kQgramPerResidue || f == kQgram || filter_is_set(f) ? -3 : 0; }
// Pattern bytes a byte-parallel kind tests (0: not byte-parallel).
constexpr __host__ __device__ int filter_bytes(Filter f)
{
    return f == kBytes1 ? 1 : f == kBytes2 ? 2 : f == kBytes3 ? 3 : f == kBytes5 ? 5 : 0;
}
// Kinds whose filter is exact for every pattern they run: no candidate is ever verified.
constexpr __host__ __device__ bool filter_never_verifies(Filter f) { return f == kShiftAnd || f == kBytes1 || f == kBytes2 || f == kBytes3; }
// The filter's candidates are the matches of an m-byte pattern: nothing to verify.
constexpr __host__ __device__ bool filter_exact(Filter f, int32_t m)
{
    return f == kShiftAnd || (filter_variant(f) == BMX_VARIANT_WINDOW && (m <= 4 || (f == kBytes5 && m == 5)));
}

// Kernel arguments (passed by value: they live in the constant bank of the launch).
struct ScanArgs {
    const uint8_t *vtext;   // 16-byte aligned base A <= text; "V space" offset v addresses A[v]
    int64_t vlen;           // lead + n: bytes of V that may be read
    int64_t vmin;           // first valid start position in V (= lead)
    int64_t vmax;           // last valid start position in V (= lead + n - m)
    int64_t pos_bias;       // reported position = v + pos_bias (= pos_base - lead)
    int32_t m;
    uint32_t num_tiles;
    uint32_t stages;        // pipeline depth
    uint32_t stage_stride;  // bytes between stages in shared memory
    uint32_t halo;          // bytes staged behind a tile
    uint32_t verify_smem;   // 1: candidates are verified from the staged tile, 0: from global
    uint32_t dense_lanes;   // a warp whose segments held candidates in this many lanes on average builds all masks right away
    uint32_t pat_smem;      // 1: pattern + tables copied to shared memory
    uint32_t coop_verify;   // 1: flagged chunks are checked by the whole warp (coop_verify16), 0: by their own lane with BM skips
    // filter constants
    uint32_t f[4];          // QGRAM: hash of P[r..r+q) for r = 0..3; WINDOW: f[0] = target
    uint32_t hmul;          // QGRAM: hash multiplier K << (32 - 8*(q-4)); the shift drops the bytes beyond the q-gram
    uint32_t hmulr[4];      // QGRAM, 7 <= m <= 10: one multiplier per residue (residue r sees min(8, m - r) bytes)
    uint32_t pad0;          // pad0, pad1: bcast and every field behind it stay at the offsets the kernels were tuned with;
                            // shifted, the byte-parallel kernels lost 0.5-0.8 % count-only (NVIDIA B200, 1000 W power limit)
    uint32_t bcast[5];      // WINDOW, byte-parallel kernels: pattern byte k replicated into the four bytes of a word
    uint32_t pad1[2];
    // per-pattern block in global memory
    const uint8_t *g_pat;
    const int32_t *g_bad;
    const int32_t *g_good;
    // output
    int64_t *pos_out;
    int64_t pos_cap;
    uint32_t *tile_counter;                // [0] tile tickets, [1] CTAs done, [2] dense-item tickets, [3] #dense blocks; zero before the launch
    uint32_t *dense_list;                  // indices of the dense blocks, ascending (written by the last CTA)
    uint16_t *mask16;                      // hit mask per chunk (written only where a segment has hits)
    uint16_t *seg_count;                   // hits per segment, zeroed before the launch
    uint32_t *block_sum;                   // hits per block, zeroed before the launch
    uint8_t *item_flag;                    // 1 if the 32 KiB work item has hits, zeroed before the launch
    unsigned long long *block_base;        // exclusive prefix of block_sum (block-scan kernel)
    uint32_t num_segs;
    uint32_t num_blocks;
    int32_t owner_offset;                  // start position of mask bit 0 relative to its chunk (-3 for QGRAM)
    const unsigned long long *carry_in;    // hits reported by earlier chained scans
    unsigned long long *carry_out;         // carry_in + hits of this scan (block-scan kernel)
    unsigned long long *count_acc;         // count-only mode: running total over the chained scans (last CTA adds scan_count)
    unsigned long long *scan_count;        // count-only mode: this scan's hits, atomically accumulated; zeroed per launch
    // multi-pattern variant (kMulti): one shared candidate table for all K patterns, staged into shared memory
    const uint32_t *g_mbits;               // bitmap over the top kMultiBitmapLog2 bits of the q-gram hash
    const uint2 *g_mtable;                 // exact table, open addressing: {hash, 0x80000000 | k << 2 | r}; y == 0: empty
    const uint2 *g_mdir;                   // per pattern: {byte offset into g_mblob, length}
    const uint8_t *g_mblob;                // the patterns, each 4-byte aligned and followed by 8 bytes of padding
    unsigned long long *mcounts;           // per-pattern hit counters (exact; zeroed by the host per search)
    uint32_t npat;
    uint32_t hmul2;                        // multiplier of the third word (grams of 9..12 bytes, m_min >= 12); 0: two-word grams
    uint32_t multi_blob_smem;              // bytes of g_mblob that fit the control block's good-suffix area (multiple of 16; 0: read from global)
    uint32_t multi_smem;                   // bytes of dynamic shared memory between the control block and the stages
    unsigned long long *host_count;        // host-mapped word: the last CTA of every scan also stores the running count there (finish() reads it without a copy)
    // find-first mode (count-only kernels): key = epoch << 47 | (2^47-1 - position), combined with atomicMax, so a
    // stale word of an earlier search never needs clearing; producers stop fetching tiles behind the best hit
    unsigned long long *first_key;
    uint32_t find_epoch;                   // 0: not a find-first scan
    uint32_t first_scan;                   // first scan of a search: carry_in / count_acc count as 0 (no memset needed)
    void *zero_ptr;                        // expand kernel: the OTHER zero-initialised scratch half, left dirty by the scan before
    uint32_t zero_vec16;                   //   this one; its first zero_vec16 16-byte words are cleared for the next scan (0: nothing)
    // dictionary variant (kDict; last, so that no field in front of them moves): the dictionary's table geometry
    uint32_t mslots_log2;                  // the exact table has 2^mslots_log2 slots
    uint32_t mtable_smem;                  // 1: the exact table is staged into shared memory, 0: read from global memory (L2)
    uint32_t mocc_log2;                    // bits of the staged "home slot occupied" array: bit (slot & (2^mocc_log2 - 1))
};

// Launch description produced by plan_scan() and consumed by launch_scan().
struct ScanLaunch {
    Filter filter;
    bool fold;              // case-insensitive instance (BMX_IGNORE_CASE)
    int tile_bytes;
    int grid;
    size_t smem_bytes;
};

// Host entry points implemented in bmx_scan.cu.
Filter choose_filter(int requested_variant, const unsigned char *pat, int32_t m);
int plan_scan(int device, Filter filter, bool fold, int32_t m, bool positions, ScanArgs *args, ScanLaunch *out);
int launch_scan(const ScanArgs &args, const ScanLaunch &launch, bool positions, void *stream);
int launch_emit(const ScanArgs &args, void *stream);
int launch_export_result(const unsigned long long *d_count, const int64_t *d_pos, int64_t pos_cap, void *d_dst, int64_t head,
                         void *stream);   // block-scan + expand (positions mode)
int launch_synth_fill(void *d_text, int64_t offset, int64_t len, uint64_t seed,
                      const unsigned char *alphabet, int32_t sigma, void *stream);

// Filter constants of a single-pattern kind (host).
void fill_filter_constants(Filter filter, const unsigned char *pat, int32_t m, ScanArgs *args);

constexpr uint32_t kHashMul = 0x9E3779B1u;
// multi-pattern candidate table
constexpr int kMultiMaxPatterns = 64;
constexpr int kMultiBitmapLog2 = 18;                                   // 2^18 bits = 32 KiB
constexpr int kMultiBitmapWords = 1 << (kMultiBitmapLog2 - 5);
constexpr int kMultiSlotsLog2 = 9;                                     // 512 slots for <= 256 (pattern, residue) entries
constexpr int kMultiSlots = 1 << kMultiSlotsLog2;
constexpr uint32_t kMultiSlotMul = 0x85EBCA6Bu;
constexpr uint32_t kHashMul2 = 0xC2B2AE3Du;
constexpr size_t kMultiSmemBytes = (size_t)kMultiBitmapWords * 4 + (size_t)kMultiSlots * 8 + (size_t)kMultiMaxPatterns * 8;
// dictionaries (bmx_dict.cu): table of the next power of two >= 8 K slots (load <= 1/2), at least kMultiSlots
constexpr int kDictMaxPatterns = 65536;
constexpr int kDictMaxOccLog2 = 15;          // the occupancy array is folded to at most 2^15 bits = 4 KiB
constexpr int kDictMaxSmemSlotsLog2 = 11;    // tables of up to 2^11 slots (16 KiB, K <= 256) are staged into shared memory
// Shared memory a kDict scan keeps in front of its stages: bitmap | occupancy bits | (table, when staged).
constexpr __host__ __device__ size_t dict_smem_bytes(uint32_t slots_log2, uint32_t table_smem, uint32_t occ_log2)
{
    return (((size_t)kMultiBitmapWords * 4 + ((size_t)1 << occ_log2) / 8 + (table_smem ? ((size_t)8 << slots_log2) : 0)) + 127) &
           ~size_t(127);
}
constexpr unsigned long long kFindMask = (1ull << 47) - 1;   // find-first keys: positions below 2^47

// ---- host helpers -------------------------------------------------------------------------
// The first min(nbytes, 4) bytes at p as a little-endian word (the q-gram hashes' view of the text).
inline uint32_t le_word(const unsigned char *p, int nbytes)
{
    uint32_t w = 0;
    for (int i = 0; i < nbytes && i < 4; ++i) w |= (uint32_t)p[i] << (8 * i);
    return w;
}
// BMX_IGNORE_CASE's fold: 'A'..'Z' -> 'a'..'z', every other byte value unchanged (Python's bytes.lower()).
inline unsigned char ascii_lower(unsigned char c) { return (unsigned)(c - 'A') < 26u ? (unsigned char)(c | 0x20u) : c; }
// Hash multiplier of a word that contributes `bytes` bytes to a gram: K << (32 - 8*bytes) drops the bytes beyond it.
inline uint32_t gram_multiplier(uint32_t K, int bytes) { return bytes >= 4 ? K : (bytes == 0 ? 0u : (K << (32 - 8 * bytes))); }
// An integer environment knob, read on every call (tests change them between calls).
inline int env_int(const char *name, int fallback)
{
    const char *v = getenv(name);
    return (v && *v) ? atoi(v) : fallback;
}

}  // namespace bmx
