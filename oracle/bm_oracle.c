/*
 * bm_oracle.c -- CPU restatement ("O2, widened") of the reference's Boyer-Moore path.
 *
 * TEST INFRASTRUCTURE ONLY (see bm_oracle.h).  Parity status: PINNED against the reference's
 * own code compiled here (oracle/_ref/libref_bm.so) and against tests/golden/golden.npz.
 *
 * Every function names the reference lines it follows.  "Reference" paths are relative to
 * /root/reference/BoyreMoore/: BoyreMoore/BoyreMoore.cpp and x64/Debug/kernel1.cl (the copy
 * the shipped exe loads; BoyreMoore/kernel1.cl does not compile and is not followed).
 */
#include "bm_oracle.h"

#include <pthread.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

/* ------------------------------------------------------------------------------------------
 * Table construction (BoyreMoore.cpp:13-68 helpers, :153-190 fill)
 * ---------------------------------------------------------------------------------------- */

/* BoyreMoore.cpp:153-162.  All 256 byte values start at m; every pattern byte except the last
 * one then records its distance to the last pattern position (later occurrences win). */
void oracle_build_bad(const unsigned char *pat, int32_t m, int32_t bad[256])
{
    for (int c = 0; c < 256; ++c)
        bad[c] = m;
    for (int32_t i = 0; i + 2 <= m; ++i)
        bad[pat[i]] = m - 1 - i;
}

/* BoyreMoore.cpp:16-28 (searchFirst).  Compares the prefix of length m-sub with the suffix
 * starting at sub. */
int32_t oracle_prefix_equals_suffix(const unsigned char *pat, int32_t m, int32_t sub)
{
    int32_t span = m - sub;
    for (int32_t t = 0; t < span; ++t)
        if (pat[t] != pat[sub + t])
            return -1;
    return 0;
}

/* BoyreMoore.cpp:30-60 (search).  Walks candidate start indices from sub-1 down to 0; a
 * candidate whose left neighbour equals P[sub-1] is skipped (:37-41); the first candidate
 * whose span bytes all equal the suffix wins (:44-57). */
int32_t oracle_suffix_reoccurrence(const unsigned char *pat, int32_t m, int32_t sub)
{
    int32_t span = m - sub;
    unsigned char before_suffix = pat[sub - 1];
    for (int32_t at = sub - 1; at >= 0; --at) {
        if (at >= 1 && pat[at - 1] == before_suffix)
            continue;
        int differs = 0;
        for (int32_t t = 0; t < span; ++t)
            if (pat[at + t] != pat[sub + t])
                differs = 1;          /* the reference keeps comparing; so do we (:47-51) */
        if (!differs)
            return at;
    }
    return -1;
}

/* BoyreMoore.cpp:165-190.  k = number of matched suffix bytes. */
void oracle_build_good(const unsigned char *pat, int32_t m, int32_t *good)
{
    if (m >= 1)
        good[0] = 0; /* reference: uninitialised, never used (kernel1.cl:29-30) */
    for (int32_t k = 1; k <= m - 1; ++k) {
        int32_t sub = m - k;
        int32_t at = oracle_suffix_reoccurrence(pat, m, sub);      /* :169 */
        if (at >= 0) {
            good[k] = sub - at;                                     /* :172 */
            continue;
        }
        int32_t shift = m;                                          /* :185-189 */
        for (int32_t s = m - k + 1; s <= m - 1; ++s) {              /* :175 */
            if (oracle_prefix_equals_suffix(pat, m, s) == 0) {
                shift = s;                                          /* :180 (result is 0) */
                break;
            }
        }
        good[k] = shift;
    }
}

/* ------------------------------------------------------------------------------------------
 * The scan (x64/Debug/kernel1.cl:1-35)
 * ---------------------------------------------------------------------------------------- */

int64_t oracle_scan_partition(const unsigned char *text, const unsigned char *pat, int32_t m,
                              int64_t start, int64_t end_incl,
                              const int32_t *good, const int32_t bad[256],
                              int64_t *pos, int64_t cap)
{
    int64_t found = 0;                       /* :5-6  occ = 0, ans[id] = 0 */
    int64_t i = start + m - 1;               /* :15   index under the LAST pattern byte */
    while (i <= end_incl) {                  /* :19 */
        int32_t k = 0;
        while (k <= m - 1 && text[i - k] == pat[m - 1 - k])   /* :21-22 right-to-left */
            ++k;
        if (k == m) {                        /* :24  report, then advance by exactly one */
            if (pos && found < cap)
                pos[found] = i - (m - 1);
            ++found;
            i += 1;
            continue;
        }
        int32_t d1 = bad[text[i]] - k;       /* :27-28  byte under the last position */
        if (d1 < 1)
            d1 = 1;
        int32_t shift = d1;                  /* :30 */
        if (k > 0) {                         /* :31 */
            int32_t d2 = good[k];            /* :29 */
            if (d2 > d1)
                shift = d2;
        }
        i += shift;                          /* :33 */
    }
    return found;
}

int oracle_search(const unsigned char *text, int64_t n, const unsigned char *pat, int32_t m,
                  int64_t *pos, int64_t cap, uint64_t *count)
{
    if (m <= 0 || n < 0 || !count || (!text && n > 0) || !pat)
        return -1;
    int32_t bad[256];
    int32_t *good = (int32_t *)malloc(sizeof(int32_t) * (size_t)m);
    if (!good)
        return -1;
    oracle_build_bad(pat, m, bad);
    oracle_build_good(pat, m, good);
    *count = (uint64_t)oracle_scan_partition(text, pat, m, 0, n - 1, good, bad, pos, cap);
    free(good);
    return 0;
}

int oracle_search_partitions(const unsigned char *text, const unsigned char *pat,
                             const int32_t *se, int32_t *ans, int32_t m, int32_t nparts)
{
    if (m <= 0 || nparts < 0 || !se || !ans || !pat)
        return -1;
    int32_t bad[256];
    int32_t *good = (int32_t *)malloc(sizeof(int32_t) * (size_t)m);
    if (!good)
        return -1;
    oracle_build_bad(pat, m, bad);
    oracle_build_good(pat, m, good);
    for (int32_t id = 0; id < nparts; ++id)          /* one work-item per range, kernel1.cl:3 */
        ans[id] = (int32_t)oracle_scan_partition(text, pat, m, se[2 * id], se[2 * id + 1],
                                                 good, bad, NULL, 0);
    free(good);
    return 0;
}

/* ------------------------------------------------------------------------------------------
 * The host's word partitioner (BoyreMoore.cpp:94-141)
 * ---------------------------------------------------------------------------------------- */

void oracle_partition_words(const char *A, int32_t P, int32_t *se)
{
    /* :94-98  the index is bumped BEFORE the space test, so a space at offset 0 is not counted
     * and the terminator itself is inspected last. */
    int64_t i = 0;
    int32_t spaces = 0;
    while (A[i++] != '\0')
        if (A[i] == ' ')
            ++spaces;

    int32_t nwords = spaces + 1;
    int32_t *wlen = (int32_t *)calloc((size_t)nwords, sizeof(int32_t));   /* :100-105 */

    /* :107-117  one word length per separator, separators are skipped one at a time. */
    i = 0;
    for (int32_t j = 0; j < nwords; ++j) {
        while (A[i] != ' ' && A[i] != '\0') {
            ++wlen[j];
            ++i;
        }
        ++i;
    }

    /* :119-141  equal word counts per range; leftover words are dropped. */
    int32_t per = nwords / P;
    int32_t next_start = 0, word0 = 0, out = 0;
    for (int32_t p = 0; p < P; ++p) {
        int32_t lo = next_start;
        int32_t hi = lo;
        for (int32_t j = word0; j < word0 + per; ++j)
            hi += wlen[j];
        word0 += per;
        hi = hi + per - 1;          /* :137  the per-1 separators inside the range */
        se[out++] = lo;             /* :138 */
        se[out++] = hi - 1;         /* :139  inclusive end */
        next_start = hi + 1;        /* :140  the separating space belongs to nobody */
    }
    free(wlen);
}

/* ------------------------------------------------------------------------------------------
 * Harness: windowed multi-threaded driver (not reference code)
 * ---------------------------------------------------------------------------------------- */

typedef struct {
    const unsigned char *text, *pat;
    const int32_t *good, *bad;
    int32_t m;
    int64_t n, window;
    int64_t nwindows;
    int64_t *next;              /* shared work counter */
    pthread_mutex_t *lock;
    int64_t **wpos;             /* per-window hit buffers (malloc'd by workers) */
    int64_t *wcount;
    int collect;
} mt_job;

static void *mt_worker(void *arg)
{
    mt_job *job = (mt_job *)arg;
    for (;;) {
        pthread_mutex_lock(job->lock);
        int64_t w = (*job->next)++;
        pthread_mutex_unlock(job->lock);
        if (w >= job->nwindows)
            break;
        int64_t lo = w * job->window;
        int64_t hi = lo + job->window;           /* exclusive bound on START positions */
        if (hi > job->n)
            hi = job->n;
        int64_t end_incl = hi - 1 + (job->m - 1); /* last byte a match owned here may touch */
        if (end_incl > job->n - 1)
            end_incl = job->n - 1;
        int64_t c = oracle_scan_partition(job->text, job->pat, job->m, lo, end_incl,
                                          job->good, job->bad, NULL, 0);
        job->wcount[w] = c;
        if (job->collect && c > 0) {
            job->wpos[w] = (int64_t *)malloc(sizeof(int64_t) * (size_t)c);
            oracle_scan_partition(job->text, job->pat, job->m, lo, end_incl,
                                  job->good, job->bad, job->wpos[w], c);
        }
    }
    return NULL;
}

int oracle_search_mt(const unsigned char *text, int64_t n, const unsigned char *pat, int32_t m,
                     int64_t *pos, int64_t cap, uint64_t *count, int32_t nthreads)
{
    if (m <= 0 || n < 0 || !count || !pat)
        return -1;
    if (nthreads <= 0) {
        long on = sysconf(_SC_NPROCESSORS_ONLN);
        nthreads = on > 0 ? (int32_t)on : 1;
    }
    if (nthreads > 256)
        nthreads = 256;
    int32_t bad[256];
    int32_t *good = (int32_t *)malloc(sizeof(int32_t) * (size_t)m);
    oracle_build_bad(pat, m, bad);
    oracle_build_good(pat, m, good);

    int64_t window = (int64_t)16 << 20;                 /* 16 MiB of start positions */
    int64_t nwindows = n > 0 ? (n + window - 1) / window : 0;
    int64_t next = 0;
    pthread_mutex_t lock = PTHREAD_MUTEX_INITIALIZER;
    mt_job job = {text, pat, good, bad, m, n, window, nwindows, &next, &lock, NULL, NULL,
                  pos != NULL};
    job.wpos = (int64_t **)calloc((size_t)(nwindows + 1), sizeof(int64_t *));
    job.wcount = (int64_t *)calloc((size_t)(nwindows + 1), sizeof(int64_t));

    pthread_t tid[256];
    int started = 0;
    for (int t = 0; t < nthreads && t < nwindows; ++t)
        if (pthread_create(&tid[started], NULL, mt_worker, &job) == 0)
            ++started;
    if (started == 0)
        mt_worker(&job);
    for (int t = 0; t < started; ++t)
        pthread_join(tid[t], NULL);

    uint64_t total = 0;
    for (int64_t w = 0; w < nwindows; ++w) {
        for (int64_t q = 0; q < job.wcount[w] && job.wpos[w]; ++q)
            if (pos && (int64_t)(total + (uint64_t)q) < cap)
                pos[total + (uint64_t)q] = job.wpos[w][q];
        total += (uint64_t)job.wcount[w];
        free(job.wpos[w]);
    }
    *count = total;
    free(job.wpos);
    free(job.wcount);
    free(good);
    return 0;
}

/* ------------------------------------------------------------------------------------------
 * Harness: independent exact matcher (not reference code)
 * ---------------------------------------------------------------------------------------- */

/* Knuth-Morris-Pratt over the whole text.  Deliberately shares nothing with the Boyer-Moore
 * restatement above or with the product's tables and filters: it is the truth those are
 * checked against.  fail[j] = length of the longest proper border of pat[0..j]. */
int oracle_kmp_search(const unsigned char *text, int64_t n, const unsigned char *pat, int32_t m,
                      int64_t *pos, int64_t cap, uint64_t *count)
{
    if (m <= 0 || n < 0 || !count || (!text && n > 0) || !pat)
        return -1;
    int32_t *fail = (int32_t *)malloc(sizeof(int32_t) * (size_t)m);
    if (!fail)
        return -1;
    fail[0] = 0;
    for (int32_t j = 1, b = 0; j < m; ++j) {
        while (b > 0 && pat[j] != pat[b])
            b = fail[b - 1];
        if (pat[j] == pat[b])
            ++b;
        fail[j] = b;
    }
    uint64_t found = 0;
    int32_t q = 0;                           /* pattern bytes matched so far */
    for (int64_t i = 0; i < n; ++i) {
        while (q > 0 && text[i] != pat[q])
            q = fail[q - 1];
        if (text[i] == pat[q])
            ++q;
        if (q == m) {
            if (pos && (int64_t)found < cap)
                pos[found] = i - (m - 1);
            ++found;
            q = fail[m - 1];
        }
    }
    *count = found;
    free(fail);
    return 0;
}

/* ------------------------------------------------------------------------------------------
 * Harness: synthetic text and position checksum
 * ---------------------------------------------------------------------------------------- */

static inline uint64_t mix64(uint64_t z)
{
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

void oracle_synth_fill(unsigned char *text, int64_t offset, int64_t len, uint64_t seed,
                       const unsigned char *alphabet, int32_t sigma)
{
    int64_t p = offset, end = offset + len;
    while (p < end) {
        uint64_t j = (uint64_t)p >> 3;
        uint64_t z = mix64(seed + (j + 1) * 0x9E3779B97F4A7C15ULL);
        int k0 = (int)(p & 7);
        for (int k = k0; k < 8 && p < end; ++k, ++p) {
            unsigned b = (unsigned)((z >> (8 * k)) & 0xFF);
            text[p - offset] = alphabet[(b * (unsigned)sigma) >> 8];
        }
    }
}

uint64_t oracle_fnv1a64_positions(const int64_t *pos, int64_t count)
{
    uint64_t h = 1469598103934665603ULL;
    for (int64_t i = 0; i < count; ++i) {
        uint64_t v = (uint64_t)pos[i];
        for (int b = 0; b < 8; ++b) {
            h ^= (v >> (8 * b)) & 0xFF;
            h *= 1099511628211ULL;
        }
    }
    return h;
}
