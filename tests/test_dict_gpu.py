"""Dictionary search (bmx_dict_*): thousands of patterns in one pass, matches as (position, pattern) pairs in text order.

The checker is a plain CPU matcher: bytes.find over every pattern, the hits merged into (p, k) order -- never the
serial Boyer-Moore oracle, which is cubic in m for long patterns.  The CPU-only tests exercise the argument checks
through the ABI (they come before any device work) and the checker's own tie order; everything else runs on the GPU.

What the cases aim at: set sizes on both sides of the shared-memory table limit (K <= 256: 2^11 slots staged; above:
the table read from global memory with the folded occupancy bits in front), the hard sets (duplicates, shared
prefixes, equal grams with different tails, patterns longer than the text, matches at both ends and across the 16 KiB
tile seams, dense text), every cap class with guard bands around both device outputs, misaligned text and a
pos_base, cross-checks against bmx_search_multi and bmx_search_ex, and reuse of handles across texts, threads and
streams."""
from __future__ import annotations

import ctypes
import random
import threading
from ctypes import byref, c_int64, c_uint64, c_void_p

import numpy as np
import pytest

ALPHA = {"dna": b"ACGT", "ascii95": bytes(range(0x20, 0x7F)), "bytes256": bytes(range(256))}
TILE = 16384                       # the set kinds scan 16 KiB tiles (bmx_scan.cu plan_scan)
SMEM_TABLE_MAX_K = 256             # 2^kDictMaxSmemSlotsLog2 slots / 8 (bmx_internal.h)


# ---------------------------------------------------------------------------------------------------------------
# CPU checker
# ---------------------------------------------------------------------------------------------------------------
def find_all(text: bytes, pat: bytes) -> list[int]:
    out, i = [], text.find(pat)
    while i >= 0:
        out.append(i)
        i = text.find(pat, i + 1)
    return out


def truth(text: bytes, pats: list[bytes]):
    """(counts uint64[K], positions int64, pattern ids int32) of every pair, sorted by position, then pattern."""
    counts = np.zeros(len(pats), dtype=np.uint64)
    ps, ks = [], []
    for k, p in enumerate(pats):
        hits = find_all(text, p)
        counts[k] = len(hits)
        ps.extend(hits)
        ks.extend([k] * len(hits))
    ps = np.asarray(ps, dtype=np.int64)
    ks = np.asarray(ks, dtype=np.int32)
    order = np.lexsort((ks, ps))
    return counts, ps[order], ks[order]


def rand_bytes(rng: random.Random, n: int, alpha: bytes) -> bytes:
    idx = np.frombuffer(rng.randbytes(n), dtype=np.uint8).astype(np.int64) % len(alpha)
    return np.frombuffer(alpha, dtype=np.uint8)[idx].tobytes()


def mixed_lengths(rng: random.Random, k: int, lo: int = 7, hi: int = 4096) -> list[int]:
    """Mostly short words, every 16th pattern long, the extremes always present."""
    ms = [rng.randint(lo, 48) if i % 16 else rng.randint(lo, hi) for i in range(k)]
    ms[0] = lo
    if k > 1:
        ms[-1] = hi
    return ms


def dictionary_for(rng: random.Random, text: bytes, ms: list[int], alpha: bytes) -> list[bytes]:
    """Three in four patterns cut from the text (they occur at least once), the rest random."""
    pats = []
    for i, m in enumerate(ms):
        if i % 4 != 3 and m <= len(text):
            at = rng.randrange(len(text) - m + 1)
            pats.append(text[at: at + m])
        else:
            pats.append(rand_bytes(rng, m, alpha))
    return pats


# ---------------------------------------------------------------------------------------------------------------
# CPU-only: argument checks and the checker
# ---------------------------------------------------------------------------------------------------------------
def test_create_rejects_bad_sets_before_any_device_work(bmx):
    lib, E = bmx._lib.load(), bmx._lib
    h = c_void_p()
    good = (ctypes.c_char_p * 2)(b"abcdefg", b"hijklmno")
    ms = (ctypes.c_int32 * 2)(7, 8)
    assert lib.bmx_dict_create(0, 2, good, ms, None) == E.BMX_E_BADARG                # no out
    assert lib.bmx_dict_create(0, 0, good, ms, byref(h)) == E.BMX_E_BADARG            # empty set
    assert lib.bmx_dict_create(0, 65537, good, ms, byref(h)) == E.BMX_E_BADARG        # more than 65536
    assert lib.bmx_dict_create(0, 2, None, ms, byref(h)) == E.BMX_E_BADARG
    assert lib.bmx_dict_create(0, 2, good, None, byref(h)) == E.BMX_E_BADARG
    for bad_m in (6, 4097, 0, -1):
        bad = (ctypes.c_int32 * 2)(7, bad_m)
        assert lib.bmx_dict_create(0, 2, good, bad, byref(h)) == E.BMX_E_BADARG
        assert "pattern 1" in lib.bmx_last_error().decode()                            # names the first bad one
    with_null = (ctypes.c_char_p * 2)(b"abcdefg", None)
    assert lib.bmx_dict_create(0, 2, with_null, ms, byref(h)) == E.BMX_E_BADARG
    assert not h.value
    rc = lib.bmx_dict_create(-1, 2, good, ms, byref(h))
    assert rc in (E.BMX_E_BADARG, E.BMX_E_NODEVICE) and not h.value
    lib.bmx_dict_destroy(None)                                                          # a no-op


def test_search_rejects_bad_arguments_before_any_device_work(bmx):
    lib, E = bmx._lib.load(), bmx._lib
    fake = ctypes.create_string_buffer(256)   # never dereferenced: every check below fails first
    d = ctypes.cast(fake, c_void_p)
    counts = (c_uint64 * 2)()
    total = c_uint64()
    pos = (ctypes.c_int64 * 4)()
    pat = (ctypes.c_int32 * 4)()
    for search in (lambda *a: lib.bmx_dict_search(*a),
                   lambda dd, t, n, p, k, cap, c, tot: lib.bmx_dict_search_device(dd, t, n, 0, p, k, cap, c, tot, None)):
        assert search(None, b"abcdefgh", 8, None, None, 0, counts, byref(total)) == E.BMX_E_BADARG      # no dictionary
        assert search(d, b"abcdefgh", 8, None, None, 0, None, byref(total)) == E.BMX_E_BADARG           # no counts
        assert search(d, b"abcdefgh", 8, None, None, 0, counts, None) == E.BMX_E_BADARG                 # no total
        assert search(d, b"abcdefgh", -1, None, None, 0, counts, byref(total)) == E.BMX_E_BADARG        # n < 0
        assert search(d, None, 8, None, None, 0, counts, byref(total)) == E.BMX_E_BADARG                # no text
        assert search(d, b"abcdefgh", 8, pos, pat, -1, counts, byref(total)) == E.BMX_E_BADARG          # cap < 0
        assert search(d, b"abcdefgh", 8, pos, None, 4, counts, byref(total)) == E.BMX_E_BADARG          # one output
        assert search(d, b"abcdefgh", 8, None, pat, 4, counts, byref(total)) == E.BMX_E_BADARG


def test_dictionary_without_a_device_fails_loudly(bmx):
    if bmx.device_count() > 0:
        pytest.skip("a CUDA device is visible")
    with pytest.raises(bmx.BmxError) as e:
        bmx.Dictionary([b"abcdefg"])
    assert e.value.code == bmx._lib.BMX_E_NODEVICE


def test_checker_orders_ties_by_pattern():
    text = b"xxabcdefghij-abcdefgh"
    pats = [b"abcdefgh", b"abcdefg", b"abcdefghij", b"abcdefg"]
    counts, ps, ks = truth(text, pats)
    assert counts.tolist() == [2, 2, 1, 2]
    assert list(zip(ps.tolist(), ks.tolist())) == [(2, 0), (2, 1), (2, 2), (2, 3), (13, 0), (13, 1), (13, 3)]


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev(bmx):
    import torch

    assert torch.cuda.is_available(), "these tests need a CUDA device"
    return torch.device("cuda:0")


def to_dev(buf: bytes, dev, misalign: int = 0):
    import torch

    a = np.frombuffer(bytes(buf), dtype=np.uint8)
    t = torch.empty(a.size + misalign + 64, dtype=torch.uint8, device=dev)
    view = t[misalign: misalign + a.size]
    if a.size:
        view.copy_(torch.from_numpy(a.copy()))
    return view


def check_both_paths(bmx, dev, text: bytes, pats: list[bytes], label, d=None):
    """Host and device entry points against the checker, every pair; returns the truth."""
    want_c, want_p, want_k = truth(text, pats)
    own = d is None
    d = d or bmx.Dictionary(pats)
    try:
        c, p, k, total = d.search(text)
        assert np.array_equal(c, want_c), (label, "host counts")
        assert total == want_p.size, (label, "host total")
        assert np.array_equal(p, want_p) and np.array_equal(k, want_k), (label, "host pairs")
        c2, p2, k2, total2 = d.search_device(to_dev(text, dev), max_matches=want_p.size + 3)
        assert np.array_equal(c2, want_c) and total2 == total, (label, "device counts")
        assert np.array_equal(p2.cpu().numpy(), want_p) and np.array_equal(k2.cpu().numpy(), want_k), (label, "device pairs")
    finally:
        if own:
            d.close()
    return want_c, want_p, want_k


@pytest.mark.gpu
@pytest.mark.parametrize("k,alpha,n", [
    (1, "dna", 1 << 20), (64, "ascii95", 1 << 20), (65, "bytes256", 1 << 20),
    (SMEM_TABLE_MAX_K, "dna", 1 << 20), (SMEM_TABLE_MAX_K + 1, "dna", 1 << 20),   # last staged table, first global one
    (1000, "ascii95", 1 << 20), (4096, "dna", 1 << 20), (65536, "bytes256", 1 << 18)])
def test_set_sizes(bmx, dev, k, alpha, n):
    rng = random.Random(k * 7919 + n)
    text = rand_bytes(rng, n, ALPHA[alpha])
    pats = dictionary_for(rng, text, mixed_lengths(rng, k, hi=min(4096, n)), ALPHA[alpha])
    c, _, _ = check_both_paths(bmx, dev, text, pats, (k, alpha))
    assert c.sum() >= (3 * k) // 4 - 1   # the cut patterns were found at least once


@pytest.mark.gpu
def test_hard_sets(bmx, dev):
    rng = random.Random(11)
    n = 5 * TILE + 1234
    base = bytearray(rand_bytes(rng, n, ALPHA["ascii95"]))
    word = b"seamless-word-0123456789"
    # matches at both ends and across every tile seam (starting 1..20 bytes in front of it)
    for at in [0, n - len(word)] + [s * TILE - rng.randint(1, 20) for s in range(1, 5)]:
        base[at: at + len(word)] = word
    text = bytes(base)
    pats = [
        word, word,                                 # duplicates: both reported
        word[:7], word[:12], word[:16], word,       # shared prefixes: ties at one start, ordered by k
        word[:12] + b"X" * 5, word[:12] + b"Y",     # equal 12-byte grams, different tails (no match)
        word[:13] + b"!" * 4,
        text[:9], text[-9:],                        # the text's first and last bytes
        text[TILE - 2000: TILE + 2096],             # 4096 bytes across the first seam
    ]
    check_both_paths(bmx, dev, text, pats, "hard")
    short = text[:3000]
    check_both_paths(bmx, dev, short, pats + [short + b"tail"], "longer than the text")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [7, 64, 20_000, 3 * TILE + 5])
def test_dense_text(bmx, dev, n):
    text = b"a" * n
    pats = [b"a" * m for m in range(7, 65)] + [b"a" * 9, b"a" * 7]   # up to 60 patterns at every start
    check_both_paths(bmx, dev, text, pats, ("dense", n))


@pytest.mark.gpu
def test_english_word_list(bmx, dev, golden):
    text = golden.text("input5L")
    words = sorted({w for w in text.split() if 7 <= len(w) <= 64})
    assert len(words) > 50
    _, p, _ = check_both_paths(bmx, dev, text, words, "english")
    assert p.size > 1000


SENT_POS, SENT_PAT, G = 0x5A5A5A5A5A5A5A5A, 0x3C3C3C3C, 16


@pytest.mark.gpu
def test_caps_write_exact_prefixes_inside_guard_bands(bmx, dev):
    import torch

    rng = random.Random(5)
    text = rand_bytes(rng, 300_000, ALPHA["dna"])
    pats = dictionary_for(rng, text, [rng.randint(7, 40) for _ in range(300)], ALPHA["dna"])
    pats += [pats[0], pats[1][:7]]   # a duplicate and a prefix: ties inside the list
    want_c, want_p, want_k = truth(text, pats)
    total = want_p.size
    assert total > 300
    lib = bmx._lib.load()
    d = bmx.Dictionary(pats)
    t = to_dev(text, dev)
    pos_base = (1 << 36) + 3
    for cap in (0, 1, total - 1, total, total + 7):
        pos_buf = torch.full((cap + 2 * G,), SENT_POS, dtype=torch.int64, device=dev)
        pat_buf = torch.full((cap + 2 * G,), SENT_PAT, dtype=torch.int32, device=dev)
        counts = np.zeros(len(pats), dtype=np.uint64)
        tot = c_uint64()
        s = torch.cuda.current_stream(dev)
        rc = lib.bmx_dict_search_device(d._h, c_void_p(t.data_ptr()), t.numel(), c_int64(pos_base),
                                        c_void_p(pos_buf.data_ptr() + 8 * G), c_void_p(pat_buf.data_ptr() + 4 * G), cap,
                                        counts.ctypes.data, byref(tot), c_void_p(s.cuda_stream))
        assert rc == 0, lib.bmx_last_error()
        assert tot.value == total and np.array_equal(counts, want_c), cap
        k = min(cap, total)
        pb, kb = pos_buf.cpu().numpy(), pat_buf.cpu().numpy()
        assert np.array_equal(pb[G: G + k], want_p[:k] + pos_base), cap
        assert np.array_equal(kb[G: G + k], want_k[:k]), cap
        assert (pb[:G] == SENT_POS).all() and (pb[G + k:] == SENT_POS).all(), cap
        assert (kb[:G] == SENT_PAT).all() and (kb[G + k:] == SENT_PAT).all(), cap
        # the host entry with the same cap
        c2, p2, k2, t2 = d.search(text, max_matches=cap)
        assert t2 == total and np.array_equal(p2, want_p[:k]) and np.array_equal(k2, want_k[:k]), cap
    d.close()


@pytest.mark.gpu
def test_misaligned_text_and_pos_base(bmx, dev):
    rng = random.Random(9)
    text = rand_bytes(rng, 70_001, ALPHA["ascii95"])
    pats = dictionary_for(rng, text, mixed_lengths(rng, 500, hi=300), ALPHA["ascii95"])
    want_c, want_p, want_k = truth(text, pats)
    d = bmx.Dictionary(pats)
    for mis in range(0, 16):
        base = mis * 1_000_003
        c, p, k, total = d.search_device(to_dev(text, dev, misalign=mis), max_matches=want_p.size, pos_base=base)
        assert np.array_equal(c, want_c) and total == want_p.size, mis
        assert np.array_equal(p.cpu().numpy(), want_p + base) and np.array_equal(k.cpu().numpy(), want_k), mis
    d.close()


@pytest.mark.gpu
def test_pairs_agree_with_search_multi_and_search(bmx, dev):
    rng = random.Random(21)
    text = rand_bytes(rng, 400_000, ALPHA["dna"])
    pats = dictionary_for(rng, text, [rng.randint(7, 64) for _ in range(64)], ALPHA["dna"])
    with_dup = pats[:63] + [pats[5]]
    d = bmx.Dictionary(with_dup)
    c, p, k, total = d.search(text)
    multi = bmx.search_multi(text, with_dup)
    for j, (cnt, plist) in enumerate(multi):
        assert c[j] == cnt and np.array_equal(p[k == j], plist), j
    d.close()

    big = dictionary_for(rng, text, mixed_lengths(rng, 3000, hi=2000), ALPHA["dna"])
    d = bmx.Dictionary(big)
    c, p, k, total = d.search_device(to_dev(text, dev), max_matches=1 << 20)
    p, k = p.cpu().numpy(), k.cpu().numpy()
    assert total == p.size
    for j in rng.sample(range(len(big)), 40):
        cnt, plist = bmx.search(text, big[j])
        assert c[j] == cnt and np.array_equal(p[k == j], plist), j
    d.close()


@pytest.mark.gpu
def test_reuse_threads_and_alternating_handles(bmx, dev):
    import torch

    rng = random.Random(33)
    texts = [rand_bytes(rng, n, ALPHA["ascii95"]) for n in (200_000, 5_000, 123_457, 0, 6)]
    pats_a = dictionary_for(rng, texts[0], mixed_lengths(rng, 700, hi=100), ALPHA["ascii95"])
    pats_b = dictionary_for(rng, texts[2], mixed_lengths(rng, 90, hi=100), ALPHA["ascii95"])
    da, db = bmx.Dictionary(pats_a), bmx.Dictionary(pats_b)
    # one handle, several texts; two handles alternating on one thread (stale counters or tables would show)
    for t in texts + texts[::-1]:
        for d, pats in ((da, pats_a), (db, pats_b)):
            check_both_paths(bmx, dev, t, pats, ("reuse", len(t), d.npat), d=d)

    # one handle, two threads, two streams
    wants = [truth(t, pats_a) for t in texts[:3]]
    errors = []

    def worker(seed):
        try:
            s = torch.cuda.Stream(dev)
            order = list(range(3)) * 3
            random.Random(seed).shuffle(order)
            for i in order:
                dt = to_dev(texts[i], dev)
                torch.cuda.current_stream(dev).synchronize()
                c, p, k, total = da.search_device(dt, max_matches=wants[i][1].size + 1, stream=s)
                ok = np.array_equal(c, wants[i][0]) and np.array_equal(p.cpu().numpy(), wants[i][1]) and \
                    np.array_equal(k.cpu().numpy(), wants[i][2])
                if not ok:
                    errors.append((seed, i))
        except Exception as e:   # reported below, in the test's thread
            errors.append((seed, repr(e)))

    threads = [threading.Thread(target=worker, args=(s,)) for s in (1, 2)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors
    da.close()
    db.close()
