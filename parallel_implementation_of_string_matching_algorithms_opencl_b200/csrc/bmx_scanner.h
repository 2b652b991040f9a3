// bmx_scanner.h -- the scanner object behind bmx_scanner_* (shared by bmx_abi.cu, bmx_exchange.cu and
// bmx_multi.cu; not installed).
#pragma once

#include <cuda_runtime.h>

#include <vector>

#include "bmx_internal.h"

struct bmx_scanner {
    int device = 0;
    // per-pattern state
    int32_t m = 0;             // pattern length (multi-pattern mode: the shortest one -- it bounds the start positions of a scan)
    int32_t m_halo = 0;        // multi-pattern mode: the longest pattern (sizes the staged halo); 0 = m
    bmx::Filter filter = bmx::kQgram;   // the scan kernel's filter kind (kMulti in multi-pattern mode)
    bool fold = false;         // case-insensitive scans (BMX_IGNORE_CASE with a pattern that has an ASCII letter): pat is folded
    cudaEvent_t ev_pat = nullptr; // recorded behind the upload of the block
    cudaStream_t pat_stream = nullptr;
    std::vector<unsigned char> pat;
    void *d_block = nullptr;  // [bad 256 x i32][good m x i32][pattern m bytes]
    size_t d_block_cap = 0;
    bmx::ScanArgs proto{};    // filter constants + pattern pointers
    // result state
    unsigned long long *d_ctrl = nullptr;  // [0],[1] carry ping-pong, [2] count-only running total, [3] always 0
    unsigned long long *h_result = nullptr;  // pinned, mapped into the device's address space
    unsigned long long *d_result = nullptr;  // device view of h_result: the last kernel of a search writes the count there
    void *d_scratch = nullptr;  // ticket, block sums/bases, segment counts, hit masks (see bmx_scanner_scan)
    size_t d_scratch_cap = 0;
    size_t zero_cap = 0;        // bytes of each of the two zero-initialised halves at the front of d_scratch
    size_t dirty[2] = {0, 0};   // leading bytes of each half that enqueued work leaves non-zero
    int cur_half = 0;           // half the next scan uses
    int64_t *d_pos_out = nullptr;
    int64_t pos_cap = 0;
    bool positions = false;
    uint32_t scan_index = 0;
    uint32_t find_epoch = 0;      // != 0: the scans of this search are find-first scans (count-only kernels, early stop)
    uint32_t find_epochs_used = 0;
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;  // around the scan kernel alone
    bool timing_open = false;
    int timing_level = 2;  // 0 none, 1 whole scan, 2 + scan kernel alone
    bmx_stats stats{};
};

namespace bmx {

// Device word holding the search's hit count: the carry slot the last scan wrote (positions mode), the
// running total (count-only mode), or the constant zero while no scan has been launched since begin().
inline const unsigned long long *result_slot(const bmx_scanner *s)
{
    if (s->scan_index == 0) return s->d_ctrl + 3;
    return s->positions ? s->d_ctrl + (s->scan_index & 1u) : s->d_ctrl + 2;
}

}  // namespace bmx
