/*
 * bm_oracle.h -- CPU restatement ("O2, widened") of the reference's Boyer-Moore path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the product: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load it,
 * and only as the checker or the reported CPU baseline.  The product path (libbmx.so) never
 * links, loads or calls anything declared here.
 *
 * Parity status: PINNED.  The restatement is checked (tests/test_oracle.py) against
 *   (1) oracle/_ref/libref_bm.so = the reference's own kernel1.cl + BoyreMoore.cpp table code
 *       compiled unmodified through a macro shim (oracle/build_oracle.sh), by fuzzing and on
 *       the reference's fixtures, and
 *   (2) golden vectors produced by that reference build (tests/golden/golden.npz, made by
 *       tests/golden/make_golden.py), which travel to the GPU box.
 * The reference itself ships no expected outputs (BoyreMoore/x64/Debug/tests.txt holds "15").
 *
 * What is "widened" relative to the reference (SURVEY.md section A.4):
 *   - text indices are int64_t (reference: int, BoyreMoore.cpp:73,86; kernel1.cl:14-15)
 *   - the bad-symbol table has 256 entries indexed by unsigned char
 *     (reference: int badSymTab[128] indexed by signed char, BoyreMoore.cpp:151,161)
 *   - the pattern buffer is sized by m (reference: char word[100], BoyreMoore.cpp:144)
 * On the reference's legal domain (7-bit bytes, n < 2^31, m <= 99) both give identical tables,
 * identical shifts and identical hit lists.
 */
#ifndef BM_ORACLE_H
#define BM_ORACLE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* BoyreMoore.cpp:153-162 -- bad-symbol table; bad[c] = m, then bad[P[i]] = m-1-i for i <= m-2. */
void oracle_build_bad(const unsigned char *pat, int32_t m, int32_t bad[256]);

/* BoyreMoore.cpp:16-28 (searchFirst) -- 0 iff P[0..m-sub) == P[sub..m), else -1. */
int32_t oracle_prefix_equals_suffix(const unsigned char *pat, int32_t m, int32_t sub);

/* BoyreMoore.cpp:30-60 (search) -- right-most i < sub where the suffix P[sub..m) re-occurs at i
 * and is not preceded by P[sub-1]; -1 if none. */
int32_t oracle_suffix_reoccurrence(const unsigned char *pat, int32_t m, int32_t sub);

/* BoyreMoore.cpp:165-190 -- good-suffix table good[1..m-1]; good[0] is set to 0 here
 * (the reference leaves it uninitialised and never uses it, kernel1.cl:29-30). */
void oracle_build_good(const unsigned char *pat, int32_t m, int32_t *good);

/* x64/Debug/kernel1.cl:1-35 -- scan of one inclusive partition [start, end_incl].
 * Writes up to cap ascending start positions into pos (may be NULL), returns the full count. */
int64_t oracle_scan_partition(const unsigned char *text, const unsigned char *pat, int32_t m,
                              int64_t start, int64_t end_incl,
                              const int32_t *good, const int32_t bad[256],
                              int64_t *pos, int64_t cap);

/* Serial reference result: tables + one partition {0, n-1}.  Returns 0, or -1 on bad args
 * (m <= 0 is rejected; the reference would report n+1 bogus hits, SURVEY.md A.6). */
int oracle_search(const unsigned char *text, int64_t n, const unsigned char *pat, int32_t m,
                  int64_t *pos, int64_t cap, uint64_t *count);

/* Argument-for-argument mirror of the kernel entry (kernel1.cl:1): nparts inclusive ranges
 * se[2*id], se[2*id+1]; ans[id] = hits fully inside range id.  Tables are rebuilt internally. */
int oracle_search_partitions(const unsigned char *text, const unsigned char *pat,
                             const int32_t *se, int32_t *ans, int32_t m, int32_t nparts);

/* BoyreMoore.cpp:94-141 -- the host's word partitioner (P ranges split on spaces).
 * Needs a NUL-terminated text like the reference (it walks until '\0').  se has 2*P ints. */
void oracle_partition_words(const char *text_nul_terminated, int32_t P, int32_t *se);

/* Windowed multi-threaded driver over oracle_scan_partition (harness, not reference code):
 * window w owns start positions [w*W, (w+1)*W) and reads (m-1) bytes of halo.  The result is
 * identical to oracle_search.  nthreads <= 0 means "all online cores". */
int oracle_search_mt(const unsigned char *text, int64_t n, const unsigned char *pat, int32_t m,
                     int64_t *pos, int64_t cap, uint64_t *count, int32_t nthreads);

/* Independent exact matcher (harness, not reference code): Knuth-Morris-Pratt, linear time, all
 * overlapping start positions ascending.  It shares no logic with the Boyer-Moore tables, the
 * q-gram filters or the kernels, so the tests use it as the truth for both the restatement and
 * the GPU path.  Writes up to cap positions into pos (may be NULL); *count is the full count.
 * Returns 0, or -1 on bad args (m <= 0). */
int oracle_kmp_search(const unsigned char *text, int64_t n, const unsigned char *pat, int32_t m,
                      int64_t *pos, int64_t cap, uint64_t *count);

/* Synthetic text shared by tests and bench (same definition as bmx_synth_fill_device):
 * 8 bytes per splitmix64 draw, word j = mix(seed + (j+1)*0x9E3779B97F4A7C15), byte k of the
 * draw b = (z >> 8k) & 0xFF is mapped to alphabet[(b * sigma) >> 8].  Fills text[0..len) with
 * the bytes at absolute offsets [offset, offset+len). */
void oracle_synth_fill(unsigned char *text, int64_t offset, int64_t len, uint64_t seed,
                       const unsigned char *alphabet, int32_t sigma);

/* FNV-1a-64 over positions, each hashed as one 64-bit unit (8 little-endian bytes). */
uint64_t oracle_fnv1a64_positions(const int64_t *pos, int64_t count);

#ifdef __cplusplus
}
#endif
#endif
