/*
 * bmx.h -- C ABI of libbmx.so, the B200-native (sm_100a) replacement for the one data-parallel
 * hot path of AnupBS28/PARALLEL_IMPLEMENTATION_OF_STRING_MATCHING_ALGORITHMS_OPENCL: the
 * partitioned Boyer-Moore text scan of BoyreMoore/.
 *
 * The reference has no plugin/FFI layer.  Its boundary is the OpenCL kernel entry
 *     search(text, pattern, se, ans, gstable, bstable, sublength)      x64/Debug/kernel1.cl:1
 * driven by the host glue in BoyreMoore/BoyreMoore/BoyreMoore.cpp:192-313 (buffers :233-252,
 * arguments :264-270, launch :273-280, read-back :286).  Every entry point below names the
 * reference lines it replaces.  "BoyreMoore.cpp" means BoyreMoore/BoyreMoore/BoyreMoore.cpp and
 * "kernel1.cl" means BoyreMoore/x64/Debug/kernel1.cl (the copy the shipped exe loads).
 *
 * Conventions
 *   - plain C types only; no torch / CUDA types (a stream travels as void* = cudaStream_t).
 *   - return 0 (BMX_OK) or a negative bmx_status; never throws; bmx_last_error() (thread-local)
 *     explains the last failure on the calling thread.
 *   - positions are 0-based byte offsets of the match START, ascending, overlapping occurrences
 *     all reported (kernel1.cl:24 advances by exactly one after a match).
 *   - the caller owns every buffer it passes; the library owns only handles it created.
 *   - there is NO CPU fallback: without a CUDA device every scanning call fails with
 *     BMX_E_NODEVICE / BMX_E_CUDA.
 */
#ifndef BMX_H
#define BMX_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BMX_VERSION 200 /* 0.2.0 */

typedef enum bmx_status {
    BMX_OK = 0,
    BMX_E_BADARG = -1,    /* NULL where data is required, m <= 0, n < 0, m > BMX_MAX_PATTERN ... */
    BMX_E_CUDA = -2,      /* a CUDA runtime call failed; see bmx_last_error() */
    BMX_E_NOMEM = -3,     /* host or device allocation failed */
    BMX_E_NODEVICE = -4,  /* no CUDA device visible */
    BMX_E_TABLES = -5,    /* caller-supplied gs/bs tables differ from the ones this pattern needs */
    BMX_E_EXCHANGE = -6   /* multi-GPU exchange step failed: no peer access, IPC mapping failed, or a peer timed out */
} bmx_status;

/* Longest supported pattern (the reference stops at 99: char word[100], BoyreMoore.cpp:144). */
#define BMX_MAX_PATTERN (1 << 20)

/* Scan variants.  AUTO picks by pattern length from measured throughput (DESIGN.md). */
typedef enum bmx_variant {
    BMX_VARIANT_AUTO = 0,
    BMX_VARIANT_QGRAM = 1,    /* m >= 7: aligned q-gram hash filter + warp ballot + warp-cooperative verify (BM-skip walk beyond m = 1024) */
    BMX_VARIANT_WINDOW = 2,   /* any m : window filter, exact for m <= 4 (m = 5 on small alphabets), else + verify */
    BMX_VARIANT_SHIFTAND = 3  /* m <= 32: bit-parallel Shift-And (the Shift-Or family) */
} bmx_variant;

/*
 * Case-insensitive search (grep -i over ASCII): OR'ed into the `variant` argument of bmx_search_ex,
 * bmx_search_device_ex and bmx_scanner_set_pattern.  Position p then matches when fold(text[p+i]) == fold(pat[i])
 * for every i < m, where fold maps 'A'..'Z' (0x41-0x5A) to 'a'..'z' and leaves every other byte value alone,
 * 0x80-0xFF included (Python's bytes.lower(); no Unicode or locale folding).  The result -- count, positions,
 * ordering, pos_cap truncation, pos_base -- is exactly the exact search's result for lower(text) and lower(pat).
 * The caller's text is never written: the scan kernel folds its own shared-memory copy of each tile.
 * An unknown bit in `variant`, or an unknown base variant with the flag, is BMX_E_BADARG.  A pattern without an
 * ASCII letter matches the same set either way: the flag is then dropped and the exact kernels run.
 * bmx_stats.variant reports `variant | BMX_IGNORE_CASE` exactly when the case-folding kernels ran.
 */
#define BMX_IGNORE_CASE 0x100

/* Per-call measurements filled by the *_ex / scanner calls (all optional). */
typedef struct bmx_stats {
    float device_ms;       /* CUDA-event time of the scan + expand kernel(s) on the launching stream */
    int32_t variant;       /* bmx_variant actually run */
    int32_t kernel_launches; /* scan kernels launched by the call */
    int32_t grid;          /* CTAs of the (last) scan kernel */
    int32_t stages;        /* TMA pipeline stages per CTA */
    int32_t tile_bytes;    /* text bytes per tile */
    int32_t smem_bytes;    /* dynamic shared memory per CTA */
    int64_t tiles;         /* tiles scanned */
    float scan_kernel_ms;  /* CUDA-event time of the (last) scan kernel alone */
    int32_t reserved;
} bmx_stats;

int bmx_version(void);
const char *bmx_last_error(void);

/* Number of visible CUDA devices (0 when there is none; never fails). */
int bmx_device_count(void);

/*
 * Device memory policy.  The convenience calls (bmx_search*, bmx_find_first*, bmx_search_partitions,
 * bmx_search_multi) keep, per calling host thread and device, one device buffer for the text and one for the
 * positions (plain cudaMalloc blocks, grown on demand, never sized by the 8-bytes-per-text-byte worst case)
 * plus pinned staging buffers, so that repeated calls do not allocate.  The library does not change any
 * attribute of the device's memory pools.  bmx_release_memory gives the calling thread's cached buffers for
 * `device` (< 0: every device) back to the driver; a host thread that exits releases everything it held.
 * (The reference allocates and releases its six cl_mem buffers on every iteration, BoyreMoore.cpp:233-244,299-310.)
 */
int bmx_release_memory(int device);

/*
 * Pattern pre-processing, once per pattern -- replaces BoyreMoore.cpp:153-162 (bad-symbol
 * table) and :165-190 with helpers :16-60 (good-suffix table).
 *   bad[c]  = m for every byte value c, then bad[P[i]] = m-1-i for i = 0..m-2  (256 entries,
 *             indexed by unsigned byte; the reference has 128 entries indexed by signed char).
 *   good[k] = the reference's strong good-suffix shift after k matched suffix bytes,
 *             k = 1..m-1; good[0] = 0 (the reference leaves it uninitialised and unused).
 * Pure host code, O(m) time; values identical to the reference's O(m^3) construction.
 */
int bmx_build_tables(const char *pat, int32_t m, int32_t bad[256], int32_t *good /* m ints */);

/*
 * Host-pointer search -- replaces the whole of BoyreMoore.cpp:192-313: device buffers,
 * host->device copies, launch, read-back.  text/pat/pos_out/count_out are HOST pointers.
 * Finds every start p in [0, n-m] with text[p..p+m) == pat, i.e. the reference's serial result
 * (one partition {0, n-1}).  *count_out is always the full count; at most pos_cap positions are
 * written (the smallest ones); pos_out may be NULL for count-only.  m > n is not an error
 * (count 0, kernel1.cl:15,19); m <= 0 is BMX_E_BADARG.  Synchronous.  The host->device copy is
 * chunked and overlapped with scanning (pinned memory is used directly, pageable memory goes
 * through pinned bounce buffers); texts of at most 4 MiB -- the size of the reference's own
 * fixtures -- take a one-stream latency path with a single synchronisation instead.
 */
int bmx_search(const char *text, int64_t n, const char *pat, int32_t m,
               int64_t *pos_out, int64_t pos_cap, uint64_t *count_out);

/* As bmx_search, on an explicit device, with variant choice and measurements.  CUDA events are recorded only
 * when stats is non-NULL (they cost ~15 us per call).  variant may carry BMX_IGNORE_CASE. */
int bmx_search_ex(int device, const char *text, int64_t n, const char *pat, int32_t m,
                  int64_t *pos_out, int64_t pos_cap, uint64_t *count_out,
                  int32_t variant, bmx_stats *stats);

/*
 * Device-resident search -- replaces BoyreMoore.cpp:258-286 (kernel creation, clSetKernelArg,
 * clEnqueueNDRangeKernel, blocking read of the counts) for text already in device memory.
 * d_text and d_pos_out are DEVICE pointers on the current device (any alignment); pat and
 * count_out are host pointers.  Launches on `stream` (cudaStream_t, NULL = default stream),
 * then waits for it to read the count back.  *device_ms (optional) receives the CUDA-event
 * time of the scan.  d_pos_out may be NULL (count-only, no output traffic).
 */
int bmx_search_device(const void *d_text, int64_t n, const char *pat, int32_t m,
                      int64_t *d_pos_out, int64_t pos_cap, uint64_t *count_out,
                      float *device_ms, void *stream);

/*
 * K patterns, ONE pass over the text (SURVEY 8f: multi-pattern batching; the reference builds its tables once per
 * pattern, BoyreMoore.cpp:150-190, and would read -- and re-send -- the text for each).  All patterns share one
 * candidate table in shared memory (a bitmap over the hash of an aligned q-gram, probed once per aligned text word
 * whatever K is; flagged words go on to an exact table and a comparison with the pattern they name), every match
 * bumps its pattern's counter, the union of all matches goes through the ordinary ordered emission and one CTA per
 * pattern splits it into K ascending lists.  Per pattern k: counts[k] (always exact) and, when pos_out &&
 * pos_out[k], the first min(counts[k], pos_cap[k]) ascending positions -- exactly what bmx_search_ex /
 * bmx_search_device returns for that pattern alone.  A pattern longer than the text counts 0.
 * Eligible for the single pass: 1 <= npat <= 64 and every pattern 7 <= m <= 4096 bytes; other sets are searched
 * pattern by pattern over the same device copy (same results).
 * bmx_search_multi: host text, copied to the device ONCE (chunked; a text larger than the device streams through
 * the ring once per pattern).  bmx_search_multi_device: d_text and the d_pos_out[k] are DEVICE pointers on the
 * current device, pats / ms / pos_cap / counts and the array d_pos_out itself are host memory; synchronous on `stream`.
 */
int bmx_search_multi(int device, const char *text, int64_t n, int32_t npat, const char *const *pats,
                     const int32_t *ms, int64_t *const *pos_out, const int64_t *pos_cap, uint64_t *counts);
int bmx_search_multi_device(const void *d_text, int64_t n, int32_t npat, const char *const *pats, const int32_t *ms,
                            int64_t *const *d_pos_out, const int64_t *pos_cap, uint64_t *counts, void *stream);

/*
 * First occurrence with early exit -- the query of the vendored CUDA sample
 * CUDA/Parallel-Programs-master/cuda/boyer-moore/boyer-moore.cu:62-86 (which leaves the index of SOME
 * occurrence in d_retval, -1 if none), made well defined: *first_out = the SMALLEST start position p with
 * text[p..p+m) == pattern, or -1.  Equal to the first entry of bmx_search's list.  The text is scanned in
 * order in growing chunks and scanning (for host text: also the host->device copies) stops after the first
 * chunk that holds a match, so an early match costs microseconds, not a pass over the text.
 * bmx_find_first: host text (pinned or pageable).  bmx_find_first_device: d_text is a DEVICE pointer,
 * work is launched on `stream` and waited for.
 */
int bmx_find_first(const char *text, int64_t n, const char *pat, int32_t m, int64_t *first_out);
int bmx_find_first_device(const void *d_text, int64_t n, const char *pat, int32_t m, int64_t *first_out,
                          void *stream);

/* As bmx_search_device with: pos_base added to every reported position (multi-GPU shards report
 * global offsets), explicit variant (may carry BMX_IGNORE_CASE), full measurements. */
int bmx_search_device_ex(const void *d_text, int64_t n, const char *pat, int32_t m,
                         int64_t pos_base, int64_t *d_pos_out, int64_t pos_cap,
                         uint64_t *count_out, int32_t variant, bmx_stats *stats, void *stream);

/*
 * Argument-for-argument mirror of the kernel entry (kernel1.cl:1; host argument order
 * BoyreMoore.cpp:264-270): text, pattern, se, ans, gstable, bstable, sublength -- plus the
 * work-item count the reference passes as global_item_size (BoyreMoore.cpp:273).
 *   se[2*id], se[2*id+1] = INCLUSIVE byte range of work-item id (BoyreMoore.cpp:119-141);
 *   ans[id] = number of occurrences lying fully inside that range (no halo: this is the
 *   reference's partitioned behaviour, seam losses included, SURVEY.md A.5).
 * All pointers are HOST pointers.  text must hold at least max(se[2*id+1])+1 bytes.
 * gs (m ints, entries 1..m-1 checked) and bs (128 ints, the reference's size) may be NULL; when
 * given they must equal the tables this pattern needs, else BMX_E_TABLES (the device scan uses
 * its own copy, so a wrong table cannot silently change the result).
 */
int bmx_search_partitions(const char *text, const char *pat, const int32_t *se, int32_t *ans,
                          const int32_t *gs, const int32_t *bs, int32_t m, int32_t nparts);

/*
 * Many ranges of one text in one call -- generalises the kernel entry search(text, pattern, se, ans, ...)
 * (kernel1.cl:1, occurrences lying fully inside each range, no halo) with the ranges the reference builds at
 * BoyreMoore.cpp:119-141, to any number of half-open ranges, with positions.  Range d = [begin[d], end[d]),
 * 0 <= begin[d] <= end[d] <= n; ranges may come in any order, overlap or be empty.
 *   counts[d]  = number of p with begin[d] <= p, p + m <= end[d], text[p..p+m) == pat: exactly what bmx_search
 *                returns for the text + begin[d] of length end[d] - begin[d] (a match across a range edge counts
 *                in no range);
 *   offsets[d] = counts[0] + ... + counts[d-1], offsets[nranges] = the total (nranges + 1 entries, always exact);
 *   pos_out    = the ranges' position lists one after the other (CSR): pos_out[offsets[d] .. offsets[d+1]) holds
 *                range d's match starts RELATIVE TO begin[d], ascending.  Only the first min(total, pos_cap)
 *                entries are written; pos_out == NULL is counts only.
 * A ragged batch held as values + offsets o[0..D] is passed as begin = o, end = o + 1, without a copy.
 * The covered bytes are scanned once with positions and every range is answered from that one ascending list
 * (binary searches + a gather), so the per-call cost is paid once per batch, not once per range.
 * bmx_search_ranges: host text, ranges and outputs; ranges are checked on the host (BMX_E_BADARG names the first
 * bad one); only [min begin, max end) crosses PCIe.  Synchronous.
 * bmx_search_ranges_device: d_text, d_begin, d_end, d_pos_out, d_counts, d_offsets are DEVICE memory on the current
 * device; the total goes to the host (*total_out).  A range outside [0, n] is found on the device and reported as
 * BMX_E_BADARG (never a fault).  Synchronous on `stream`.
 */
int bmx_search_ranges(int device, const char *text, int64_t n, int64_t nranges,
                      const int64_t *begin, const int64_t *end, const char *pat, int32_t m,
                      int64_t *pos_out, int64_t pos_cap, uint64_t *counts, int64_t *offsets /* nranges+1 */);
int bmx_search_ranges_device(const void *d_text, int64_t n, int64_t nranges,
                             const int64_t *d_begin, const int64_t *d_end, const char *pat, int32_t m,
                             int64_t *d_pos_out, int64_t pos_cap, uint64_t *d_counts, int64_t *d_offsets,
                             uint64_t *total_out, void *stream);

/*
 * Dictionary search (grep -F -f wordlist): up to 65536 fixed strings in ONE pass over the text, matches reported in
 * text order as (position, pattern) pairs.  bmx_dict_create hashes the set once into a device block the handle owns
 * (the candidate table of bmx_search_multi, sized by the set: DESIGN §3.11); every search reuses it.
 *   create     1 <= npat <= 65536 patterns, each 7 <= ms[k] <= 4096 bytes (BMX_E_BADARG otherwise, naming the
 *              first bad one).  The handle lives on `device`, is immutable after create and may be used from
 *              several host threads at once, each with its own stream; scratch comes from the calling thread's
 *              context, as for every other entry point.
 *   result     a match is a pair (p, k) with text[p..p+ms[k]) == pats[k]; overlapping matches count.  The list of
 *              all pairs is sorted by p, then by k (patterns sharing a prefix, and duplicate patterns, tie at one p:
 *              every duplicate is reported).  counts[k] (host, npat entries) = pairs of pattern k, always exact;
 *              *total_out = their sum.  pos_out[i], pat_out[i] for i < min(total, cap) are exactly the first
 *              min(total, cap) pairs, positions with pos_base added.  The pairs of pattern k are what bmx_search_ex
 *              returns for that pattern alone (and, for npat <= 64, what bmx_search_multi returns for k).
 * bmx_dict_search_device: d_text, d_pos_out, d_pat_out are DEVICE memory on the dictionary's device (both outputs
 * NULL: counts only); synchronous on `stream`.  bmx_dict_search: host text, copied to the device once (a text that
 * does not fit there is BMX_E_NOMEM); outputs in host memory.
 */
typedef struct bmx_dict bmx_dict;
int bmx_dict_create(int device, int32_t npat, const char *const *pats, const int32_t *ms, bmx_dict **out);
void bmx_dict_destroy(bmx_dict *d);
int bmx_dict_search_device(const bmx_dict *d, const void *d_text, int64_t n, int64_t pos_base,
                           int64_t *d_pos_out, int32_t *d_pat_out, int64_t cap,
                           uint64_t *counts, uint64_t *total_out, void *stream);
int bmx_dict_search(const bmx_dict *d, const char *text, int64_t n,
                    int64_t *pos_out, int32_t *pat_out, int64_t cap, uint64_t *counts, uint64_t *total_out);

/*
 * The reference's host-side word partitioner -- replaces BoyreMoore.cpp:94-141.  Splits
 * text[0..n) (up to the first NUL, like the reference's strcpy'd copy, :89-90) on single spaces
 * into nparts inclusive byte ranges of equal word count: se[2*p], se[2*p+1].  The space between
 * two ranges belongs to neither; left-over words are dropped.  Pure host code.  Only needed to
 * feed bmx_search_partitions the numbers the reference would have used; the scan itself tiles
 * the text with an (m-1)-byte halo instead.
 */
int bmx_partition_words(const char *text, int64_t n, int32_t nparts, int32_t *se /* 2*nparts */);

/*
 * Reusable scanner: keeps the per-pattern device block (pattern, tables, filter constants), the
 * look-back scratch and the events across calls, and exposes the asynchronous pieces so a caller
 * can chain chunk scans on its own stream (this is what bmx_search builds on).
 * One scanner per host thread / stream; scanners are independent of each other.
 */
typedef struct bmx_scanner bmx_scanner;

int bmx_scanner_create(int device, bmx_scanner **out);
void bmx_scanner_destroy(bmx_scanner *s);

/* Builds the tables (bmx_build_tables) and uploads the pattern block on `stream`.  With BMX_IGNORE_CASE in
 * variant, the folded pattern's tables and block; the following scans of this scanner are case-insensitive. */
int bmx_scanner_set_pattern(bmx_scanner *s, const char *pat, int32_t m, int32_t variant, void *stream);

/* Starts a new result: zeroes the running count.  Positions of later bmx_scanner_scan calls are
 * appended to d_pos_out in call order (so scanning consecutive chunks left to right keeps the
 * list ascending). */
int bmx_scanner_begin(bmx_scanner *s, int64_t *d_pos_out, int64_t pos_cap, void *stream);

/* Asynchronously scans d_text[0..n) for matches STARTING in [0, n-m]; reports start + pos_base.
 * No host synchronisation. */
int bmx_scanner_scan(bmx_scanner *s, const void *d_text, int64_t n, int64_t pos_base, void *stream);

/* CUDA-event instrumentation of bmx_scanner_scan: 0 = none, 1 = the whole scan (device_ms), 2 = also the
 * scan kernel alone (scan_kernel_ms; default).  Event records between back-to-back kernels cost about 10 us
 * per scan on B200, so a throughput pipeline switches them off. */
int bmx_scanner_set_timing(bmx_scanner *s, int level);

/* Asynchronously packs the result for a collective into DEVICE memory d_dst on `stream`:
 * d_dst[0] = running count, d_dst[1] = positions actually written = min(count, pos_cap),
 * d_dst[2 .. 2+head) = the first `head` entries of the position buffer (entries beyond d_dst[1]
 * are unspecified).  Lets a multi-GPU caller feed the count exchange (all-reduce / all-gather)
 * without a host round trip between the scan and the collectives. */
int bmx_scanner_export_result(bmx_scanner *s, void *d_dst /* int64[2 + head] */, int64_t head, void *stream);

/* Waits for `stream`, returns the running count and (optional) statistics of the scans since
 * bmx_scanner_begin. */
int bmx_scanner_finish(bmx_scanner *s, uint64_t *count_out, bmx_stats *stats, void *stream);

/*
 * Single-process multi-GPU search over HOST text (the reference has one device, BoyreMoore.cpp:217-219, and
 * splits its text into word ranges WITHOUT overlap, :119-141).  GPU r of R receives the bytes
 * [lo_r, hi_r + m - 1): it owns the match START positions [lo_r, hi_r) and reads an (m-1)-byte halo, so an
 * occurrence straddling a seam is reported exactly once, with its global offset.  One host thread per GPU
 * drives the chunked, overlapped ingest of its shard (every GPU uses its own PCIe link); counts are summed on
 * the host and the per-shard lists are copied into pos_out in shard order, which is ascending.
 * shard_counts (optional, ngpus entries) receives the per-GPU hit counts.  Same result as bmx_search.
 * (One process per GPU with NCCL collectives is the other supported layout: distributed.py.)
 */
typedef struct bmx_mg bmx_mg;
int bmx_mg_create(int ngpus /* <= 0: all visible GPUs */, bmx_mg **out);
void bmx_mg_destroy(bmx_mg *mg);
int bmx_mg_device_count(const bmx_mg *mg);
int bmx_mg_search(bmx_mg *mg, const char *text, int64_t n, const char *pat, int32_t m,
                  int64_t *pos_out, int64_t pos_cap, uint64_t *count_out, uint64_t *shard_counts);

/*
 * The exchange step of the sharded scan (SURVEY 8e), inside the library, over NVLink peer memory -- no NCCL
 * kernel, no host synchronisation per step.  The reference has nothing of the kind: one device
 * (BoyreMoore.cpp:217-219), word ranges without overlap (:119-141), per-range counts read back with a blocking
 * clEnqueueReadBuffer (:286).
 *
 * One bmx_exchange per rank (= GPU).  Every rank owns a small device "mailbox"; bmx_exchange_post stores this
 * rank's {count, list head} into the mailboxes of its peers with plain stores through peer pointers and
 * publishes the step number behind a system-scope release; bmx_exchange_collect waits (on the device) for the
 * world's step numbers, sums the counts and -- on rank dst -- concatenates the position lists in rank order
 * (= ascending order) into d_out.  Both calls only enqueue a kernel on `stream`; bmx_exchange_wait polls a
 * host-mapped result word, it performs no CUDA call on the fast path.
 *
 * Ranks may be threads of one process (bmx_exchange_connect_local; peer access is enabled as needed) or one
 * process per GPU (torchrun): each rank publishes bmx_exchange_handle (a cudaIpcMemHandle, 64 bytes), the
 * handles travel by any means (distributed.py uses one torch.distributed all_gather at set-up) and
 * bmx_exchange_connect maps them.  head_cap positions per rank ride along with the header (ring of `depth`
 * steps); longer lists use the tail areas (two of tail_cap positions per source, alternating, on dst only).  The
 * gathered list is always a prefix of the global ascending list: it ends behind the first rank whose list did
 * not fit (its own pos_cap, or head_cap + tail_cap); the total count is exact regardless.
 *
 * Call order per rank and step: bmx_scanner_begin/scan ... -> bmx_exchange_post -> (later) bmx_exchange_collect;
 * at most depth-1 steps (with tail_cap > 0: at most 2) may be posted and not yet collected.  Collecting step q-1 after posting step q keeps
 * every GPU from ever waiting for a peer.  Device-side waits time out after BMX_XCHG_TIMEOUT_MS (default
 * 20000) and surface as BMX_E_EXCHANGE from bmx_exchange_wait.  All ranks must be connected before the first
 * post and idle before any rank is destroyed (a barrier of the caller's choice).
 */
#define BMX_EXCHANGE_HANDLE_BYTES 64
#define BMX_EXCHANGE_MAX_RANKS 16
typedef struct bmx_exchange bmx_exchange;
int bmx_exchange_create(int device, int rank, int world, int dst, int64_t head_cap, int64_t tail_cap, int depth,
                        bmx_exchange **out);
void bmx_exchange_destroy(bmx_exchange *x);
int bmx_exchange_handle(bmx_exchange *x, void *handle_out /* BMX_EXCHANGE_HANDLE_BYTES */);
int bmx_exchange_connect(bmx_exchange *x, const void *handles /* world x BMX_EXCHANGE_HANDLE_BYTES, rank order */);
int bmx_exchange_connect_local(bmx_exchange *const *all /* world exchanges of this process, rank order */, int world);
/* Ships the running result of `s` (count + the positions it holds) as the next step; *seq_out = its number (1, 2, ...). */
int bmx_exchange_post(bmx_exchange *x, bmx_scanner *s, void *stream, uint64_t *seq_out);
/* Completes the oldest uncollected step; d_out/out_cap (DEVICE memory) are used on rank dst only. */
int bmx_exchange_collect(bmx_exchange *x, int64_t *d_out, int64_t out_cap, void *stream, uint64_t *seq_out);
/* Blocks the calling host thread until step `seq` has been collected on this rank.  counts_out: world entries. */
int bmx_exchange_wait(bmx_exchange *x, uint64_t seq, uint64_t *total_out, uint64_t *counts_out, int64_t *gathered_out);

/*
 * Device-resident multi-GPU search (BASELINE config 5 from C): shard r lives on GPU r of `mg` as
 * d_text[r][0 .. n[r]) = its own start positions plus the (m-1)-byte halo, pos_base[r] = global offset of its
 * first byte.  Every GPU scans its shard, the exchange step above combines the counts and gathers the lists on
 * GPU 0 of `mg`: d_pos_out (DEVICE memory on that GPU, may be NULL) receives the first min(count, pos_cap)
 * global positions, ascending.  shard_counts (optional): ngpus entries.  Synchronous.
 */
int bmx_mg_search_device(bmx_mg *mg, const void *const *d_text, const int64_t *n, const int64_t *pos_base,
                         const char *pat, int32_t m, int64_t *d_pos_out, int64_t pos_cap, uint64_t *count_out,
                         uint64_t *shard_counts);

/*
 * Synthetic text generator used by the tests and bench.py (identical definition on the CPU in
 * oracle/bm_oracle.c:oracle_synth_fill): fills d_text[0..len) with the bytes at absolute
 * offsets [offset, offset+len) of the stream defined by (seed, alphabet[sigma]).
 * Not part of the reference; it exists so that 4 GiB .. 64 GiB inputs never cross PCIe.
 */
int bmx_synth_fill_device(void *d_text, int64_t offset, int64_t len, uint64_t seed,
                          const unsigned char *alphabet, int32_t sigma, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BMX_H */
