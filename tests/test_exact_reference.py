"""CPU: an exact matcher that shares no logic with Boyer-Moore (oracle_kmp_search, Knuth-Morris-Pratt) checked
against brute force, and then used as the truth for
  - the oracle's restatement of the reference (its own tables and skips) beyond the tiny sizes it was fuzzed at, on
    periodic patterns, patterns with long borders and near-miss texts where the good-suffix shift decides, and
  - the library's O(m) tables (bmx_build_tables) driving the reference's skip walk at the pattern lengths only the
    GPU path uses (m > 1024): the walk the kernels' lane verifier performs, so a shift that is too large shows here
    as a missed occurrence.
No GPU needed."""
from __future__ import annotations

import ctypes
import random

import numpy as np
import pytest


def kmp(oracle, text, pat: bytes) -> np.ndarray:
    """All overlapping occurrences of pat in text (bytes or uint8 array), ascending, from the KMP matcher."""
    buf = np.ascontiguousarray(np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray)) else text,
                               dtype=np.uint8)
    pat = bytes(pat)
    lib = oracle.lib
    cnt = ctypes.c_uint64()
    tp = ctypes.c_void_p(buf.ctypes.data) if buf.size else None
    rc = lib.oracle_kmp_search(tp, ctypes.c_int64(buf.size), ctypes.c_char_p(pat), ctypes.c_int32(len(pat)),
                               None, ctypes.c_int64(0), ctypes.byref(cnt))
    assert rc == 0, rc
    pos = np.zeros(max(cnt.value, 1), dtype=np.int64)
    rc = lib.oracle_kmp_search(tp, ctypes.c_int64(buf.size), ctypes.c_char_p(pat), ctypes.c_int32(len(pat)),
                               pos.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(pos.size), ctypes.byref(cnt))
    assert rc == 0, rc
    return pos[: cnt.value]


def adversarial_cases(m: int, rng: np.random.Generator, scale: int):
    """(name, text, pattern) triples built to stress Boyer-Moore skips for a pattern of m bytes.  Texts hold about
    `scale` bytes of background plus the planted copies.  Full matches are kept to a few dozen per text so that the
    right-to-left walk (m compares per match) stays cheap at m = 2^20."""
    def rand(n, sigma):
        return rng.integers(97, 97 + sigma, size=n, dtype=np.uint8)

    def rep(u, n):
        return np.resize(u, n)

    out = []
    # periodic pattern u^k: a run of u holding a few dozen occurrences, inside random text over the same letters
    for ul in (1, 2, 3, 5):
        u = rand(ul, 2)
        u[-1] = 98 if u[0] == 97 else 97 if ul > 1 else u[-1]
        pat = rep(u, m)
        run = rep(u, m + 40 * ul + int(rng.integers(0, ul)))
        out.append((f"periodic{ul}", np.concatenate([rand(scale // 2, 2), run, rand(scale // 2, 2)]), pat))
    # long borders u^k v u^j: the text repeats the same structure with the v's at slightly varying distances, so
    # many alignments match a long suffix and then fail
    for ul, vl in ((1, 1), (2, 1), (3, 2)):
        u = rand(ul, 2)
        v = (u[:vl] if vl <= ul else rand(vl, 2)) ^ 3      # differs from u in every byte
        j = max(1, (m - vl) // (3 * ul))
        k = max(0, (m - vl - j * ul + ul - 1) // ul)
        pat = np.concatenate([rep(u, k * ul), v, rep(u, j * ul)])[-m:] if k * ul + vl + j * ul >= m else None
        if pat is None or pat.size != m:
            continue
        pieces = [rand(scale // 4, 2)]
        for rep_i in range(12):
            d = int(rng.integers(-2, 3)) * ul
            pieces += [rep(u, max(ul, k * ul + d)), v]
            if rep_i % 4 == 3:
                pieces.append(pat)
        pieces += [rep(u, j * ul), rand(scale // 4, 2)]
        out.append((f"border{ul}{vl}", np.concatenate(pieces), pat))
    # near misses: copies of the pattern with one byte changed at 0, 1, m/2, m-2 or m-1 (a mismatch after a long
    # matched suffix, so the good-suffix shift decides), each followed by a true copy overlapping it at a small
    # distance or at a border distance, on random text over 2 and 4 letters
    for sigma in (2, 4):
        pat = rand(m, sigma)
        if rng.random() < 0.5:                               # self-similar: the pattern's second half repeats its first
            half = m // 2
            pat[m - half:] = pat[:half]
        text = rand(scale, sigma)
        spots = np.linspace(0, max(0, scale - 3 * m), num=12, dtype=np.int64) if scale > 3 * m else [0]
        idxs = sorted({0, 1, m // 2, max(0, m - 2), m - 1})
        pieces, at = [], 0
        for s_i, spot in enumerate(spots):
            j = idxs[s_i % len(idxs)]
            near = pat.copy()
            near[j] = near[j] ^ 1
            d = [1, 2, 3, m // 2, m - 1, m, m + 1][s_i % 7]
            region = np.concatenate([near, rand(max(0, d - m), sigma), pat]) if d >= m else None
            if region is None:
                region = near.copy()
                region = np.concatenate([region, np.zeros(d, dtype=np.uint8)])
                region[d:d + m] = pat
            pieces.append(text[at:spot] if spot >= at else np.zeros(0, dtype=np.uint8))
            pieces.append(region)
            at = max(at, int(spot))
        pieces.append(text[at:])
        out.append((f"nearmiss{sigma}", np.concatenate(pieces), pat))
    # the text is the pattern, and the pattern minus its last byte (m = n and m = n + 1)
    pat = rand(m, 2)
    out.append(("exact", pat.copy(), pat))
    out.append(("short", pat[:-1].copy(), pat))
    return out


def test_kmp_equals_brute_force(oracle):
    """The checker itself: thousands of small cases, alphabets of 1..4 symbols, every m from 1 to n + 1."""
    rnd = random.Random(7)
    for it in range(4000):
        sigma = rnd.randint(1, 4)
        n = rnd.randint(0, 60)
        text = bytes(rnd.randrange(97, 97 + sigma) for _ in range(n))
        m = rnd.randint(1, n + 1)
        if n >= m and rnd.random() < 0.5:
            o = rnd.randint(0, n - m)
            pat = text[o:o + m]
        else:
            pat = bytes(rnd.randrange(97, 97 + sigma) for _ in range(m))
        by_find, i = [], text.find(pat)
        while i >= 0:
            by_find.append(i)
            i = text.find(pat, i + 1)
        by_slice = [i for i in range(n - m + 1) if text[i:i + m] == pat]
        got = kmp(oracle, text, pat)
        assert by_find == by_slice
        assert got.tolist() == by_slice, (it, text, pat)
    # a 1 MiB text of one letter: every start matches, positions are 0..n-m
    big = np.full(1 << 20, 97, dtype=np.uint8)
    assert np.array_equal(kmp(oracle, big, b"a" * 300), np.arange(big.size - 299))
    with pytest.raises(AssertionError):
        kmp(oracle, b"abc", b"")                                         # empty pattern: rejected (-1)


@pytest.mark.parametrize("seed", range(3))
def test_oracle_restatement_equals_kmp_on_adversarial_inputs(oracle, seed):
    """The restated reference (its O(m^3) tables, right-to-left compare, bad-symbol and good-suffix skips) finds
    exactly the KMP occurrences for m from 13 to 300 -- it is correct, not just consistent with the kernels."""
    rng = np.random.default_rng(100 + seed)
    for m in (13, 16, 31, 64, 99, 100, 137, 255, 300):
        for name, text, pat in adversarial_cases(m, rng, scale=4 * m + 500):
            want = kmp(oracle, text, pat.tobytes())
            got = oracle.search(text.tobytes(), pat.tobytes())
            assert np.array_equal(got, want), (seed, m, name)
    rnd = random.Random(seed)                                            # small m, many cases of every shape
    for it in range(400):
        m = rnd.randint(2, 40)
        for name, text, pat in adversarial_cases(m, rng, scale=rnd.randint(m, 300)):
            assert np.array_equal(oracle.search(text.tobytes(), pat.tobytes()), kmp(oracle, text, pat.tobytes())), (it, m, name)


def _skip_walk(oracle, text: np.ndarray, pat: bytes, bad: np.ndarray, good: np.ndarray) -> np.ndarray:
    """oracle_scan_partition over the whole text with the given tables (the reference's skip walk)."""
    text = np.ascontiguousarray(text, dtype=np.uint8)
    n, m = text.size, len(pat)
    bad = np.ascontiguousarray(bad, dtype=np.int32)
    good = np.ascontiguousarray(good, dtype=np.int32)
    fn = oracle.lib.oracle_scan_partition
    fn.restype = ctypes.c_int64
    args = (ctypes.c_void_p(text.ctypes.data), ctypes.c_char_p(pat), ctypes.c_int32(m), ctypes.c_int64(0),
            ctypes.c_int64(n - 1), good.ctypes.data_as(ctypes.c_void_p), bad.ctypes.data_as(ctypes.c_void_p))
    count = fn(*args, None, ctypes.c_int64(0))
    pos = np.zeros(max(count, 1), dtype=np.int64)
    assert fn(*args, pos.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(pos.size)) == count
    return pos[:count]


@pytest.mark.parametrize("m", [1025, 2048, 4097, 10_000, 70_000, 1 << 20])
def test_library_tables_skip_safely_at_gpu_only_lengths(bmx, oracle, m):
    """Patterns longer than 1024 bytes are verified on the GPU only by the lane walk with the library's O(m) tables
    (the oracle's O(m^3) construction does not finish at these lengths).  The same walk on the CPU, with the same
    tables, must find every KMP occurrence on the adversarial shapes: a good-suffix or bad-symbol shift one too
    large loses matches here."""
    rng = np.random.default_rng(m)
    scale = min(6 * m, 8 << 20)
    for name, text, pat in adversarial_cases(m, rng, scale=scale):
        p = pat.tobytes()
        bad, good = bmx.build_tables(p)
        want = kmp(oracle, text, p)
        got = _skip_walk(oracle, text, p, bad, good)
        assert np.array_equal(got, want), (m, name, got.size, want.size)
