"""GPU: every kernel instance and knob-selected branch driven on purpose, with the KMP matcher
(oracle_kmp_search, no Boyer-Moore logic) as the truth.  Each case checks the full position list, capped lists
(half the count and one entry), count-only mode and find_first_device, on an aligned and an odd-offset copy of
the text.  The knobs are environment variables: BMX_QGRAM_UNIFORM and BMX_WINDOW5 are read when the pattern is set
(choose_filter), the others by plan_scan on every scan."""
from __future__ import annotations

import random
import zlib

import numpy as np
import pytest

from test_exact_reference import adversarial_cases, kmp
from test_parity_gpu import dev, to_dev  # noqa: F401  (dev is a fixture)

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

MISALIGN = (0, 5)


def set_knobs(monkeypatch, **knobs):
    for k, v in knobs.items():
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, str(v))


def check(bmx, td, pat: bytes, want: np.ndarray, variant="auto", tag=(), first=True):
    """Full list, caps of half the count and of 1, count-only and (optionally) find_first against `want`."""
    count, pos, stats = bmx.search_device(td, pat, max_positions=max(want.size, 1), variant=variant)
    assert count == want.size and np.array_equal(pos.cpu().numpy(), want), (*tag, "full", count, want.size)
    for cap in sorted({max(want.size // 2, 1), 1}):
        count, pos, _ = bmx.search_device(td, pat, max_positions=cap, variant=variant)
        assert count == want.size and np.array_equal(pos.cpu().numpy(), want[:cap]), (*tag, "cap", cap)
    count, pos, _ = bmx.search_device(td, pat, variant=variant)
    assert count == want.size and pos is None, (*tag, "count-only", count, want.size)
    if first:
        assert bmx.find_first_device(td, pat) == (int(want[0]) if want.size else -1), (*tag, "find_first")
    return stats


# ---------------------------------------------------------------------------------------------------------------
# 1. Forced emission paths: every scan-kernel instance, both tile sizes, dense-lane and verification knobs
# ---------------------------------------------------------------------------------------------------------------
# (label, variant, m, distinct bytes in the pattern's period, knobs that select the instance)
INSTANCES = [
    ("window-flag2", "window", 1, 1, {}),
    ("window-flag3", "window", 2, 2, {}),
    ("window-flag4", "window", 3, 3, {}),
    ("window-flag1-m4", "window", 4, 3, {}),
    ("window-flag1-m7", "window", 7, 3, {}),
    ("window-flag1-m16", "window", 16, 5, {}),
    ("window-flag1-m40", "window", 40, 7, {}),
    ("window-flag1-m5", "window", 5, 3, {"BMX_WINDOW5": 0}),
    ("window-flag1-m6", "window", 6, 4, {"BMX_WINDOW5": 0}),
    ("window-flag6-m5", "window", 5, 3, {"BMX_WINDOW5": 1}),
    ("window-flag6-m5-wide", "window", 5, 6, {"BMX_WINDOW5": 1}),     # > 4 distinct bytes: not chosen unforced
    ("window-flag6-m6-wide", "window", 6, 6, {"BMX_WINDOW5": 1}),
    ("qgram-flag0-m7", "qgram", 7, 3, {"BMX_QGRAM_UNIFORM": 0}),
    ("qgram-flag0-m8", "qgram", 8, 5, {"BMX_QGRAM_UNIFORM": 0}),
    ("qgram-flag0-m9", "qgram", 9, 4, {"BMX_QGRAM_UNIFORM": 0}),
    ("qgram-flag1-m7", "qgram", 7, 5, {"BMX_QGRAM_UNIFORM": 1}),
    ("qgram-flag1-m13", "qgram", 13, 6, {"BMX_QGRAM_UNIFORM": 1}),
    ("qgram-flag1-m64", "qgram", 64, 7, {"BMX_QGRAM_UNIFORM": 1}),
    ("shiftand-m1", "shiftand", 1, 1, {}),
    ("shiftand-m9", "shiftand", 9, 4, {}),
    ("shiftand-m32", "shiftand", 32, 7, {}),
]


def verifies(variant: str, m: int, knobs: dict) -> bool:
    """Whether the instance checks its candidates (the same rule as filter_exact)."""
    if variant == "shiftand" or (variant == "window" and m <= 4):
        return False
    return not (variant == "window" and m == 5 and knobs.get("BMX_WINDOW5") == 1)


def instance_texts(rng, unit: np.ndarray, pat: np.ndarray):
    """sparse random bytes256, random over four letters of the pattern, purely periodic, and mixed: 2 MiB blocks
    that alternate between the periodic text and random bytes, so a warp's dense mode flips across tiles.
    The periodic text repeats the pattern's period (at most 7 bytes), so every lane has a candidate start in each of
    its 16-position slabs of every segment: with BMX_DENSE_LANES=1 each warp is certain to run the dense path from
    its second tile on (dense-path entry is not visible in the stats)."""
    m = pat.size
    near = pat.copy()
    near[-1] ^= 1                                                       # the last byte differs
    near0 = pat.copy()
    near0[0] ^= 1

    def plant(text):
        n = text.size
        spots = [0, n - m] + [s + d for s in range(16384, n - 2 * m, 16384 * 7) for d in (-m, -(m // 2) - 1, -1, 0)]
        for k, s in enumerate(spots):
            if 0 <= s <= n - m:
                text[s:s + m] = pat
            d = s + m + 100 + k
            if 0 <= d <= n - 2 * m - 200:
                text[d:d + m] = near if k % 2 else near0
        return text

    n = (1 << 20) + 13
    sparse = plant(rng.integers(0, 256, size=n, dtype=np.uint8))
    letters = np.unique(pat)[:4]
    while letters.size < 4:
        letters = np.unique(np.concatenate([letters, rng.integers(0, 256, size=1, dtype=np.uint8)]))
    small = plant(letters[rng.integers(0, 4, size=n)].astype(np.uint8))
    periodic = np.resize(unit, n + 3)
    mixed = rng.integers(0, 256, size=(6 << 20) + 99, dtype=np.uint8)
    for b in range(0, mixed.size, 4 << 20):                            # dense, sparse, dense
        e = min(b + (2 << 20), mixed.size)
        mixed[b:e] = np.resize(unit, e - b)
    return [("bytes256", sparse), ("four-letter", small), ("periodic", periodic), ("mixed", plant(mixed))]


@pytest.mark.parametrize("label,variant,m,distinct,knobs", INSTANCES, ids=[i[0] for i in INSTANCES])
def test_forced_emission_paths(bmx, oracle, dev, monkeypatch, label, variant, m, distinct, knobs):  # noqa: F811
    rng = np.random.default_rng(zlib.crc32(label.encode()))
    unit = rng.choice(np.arange(256, dtype=np.uint8), size=distinct, replace=False)
    pat_arr = np.resize(unit, m)
    pat = pat_arr.tobytes()
    set_knobs(monkeypatch, **knobs)
    coops = (1, 0) if verifies(variant, m, knobs) else (None,)
    for tname, text in instance_texts(rng, unit, pat_arr):
        want = kmp(oracle, text, pat)
        assert want.size >= 2, (label, tname)
        for mis in MISALIGN:
            td = to_dev(text, dev, misalign=mis)
            for tile in (16384, 32768):
                for dense in (1, 33, None):
                    for coop in coops:
                        set_knobs(monkeypatch, BMX_TILE=tile, BMX_DENSE_LANES=dense, BMX_COOP_VERIFY=coop)
                        stats = check(bmx, td, pat, want, variant, (label, tname, mis, tile, dense, coop),
                                      first=dense != 33)
                        assert stats["variant"] == variant and stats["tile_bytes"] == tile
            del td


def test_one_cta_grid(bmx, oracle, dev, monkeypatch):  # noqa: F811
    """The whole text through a single CTA (every SM but one spared, one CTA per SM)."""
    rng = np.random.default_rng(3)
    unit = np.frombuffer(b"xyzzy", dtype=np.uint8)
    pat_arr = np.resize(unit, 13)
    set_knobs(monkeypatch, BMX_CTAS_PER_SM=1, BMX_SPARE_SMS=1000)
    for tname, text in instance_texts(rng, unit, pat_arr):
        want = kmp(oracle, text, pat_arr.tobytes())
        td = to_dev(text, dev, misalign=7)
        for variant in ("qgram", "window", "shiftand"):
            for dense in (1, None):
                set_knobs(monkeypatch, BMX_DENSE_LANES=dense)
                stats = check(bmx, td, pat_arr.tobytes(), want, variant, ("one-cta", tname, variant, dense))
                assert stats["grid"] == 1


# ---------------------------------------------------------------------------------------------------------------
# 2. Long patterns (pattern and window beyond shared memory) on dense and adversarial text
# ---------------------------------------------------------------------------------------------------------------
LONG_MS = [1024, 1025, 2048, 4095, 4096, 4097, 16384, 32767, 32768, 32769, 70000]


def long_pattern_texts(rng, m: int):
    """(name, text, pattern) for one pattern length: dense periodic texts, the adversarial shapes of the CPU tests,
    copies straddling 16/32 KiB tile seams (spanning three or more tiles when m > 32 KiB), m = n and m = n - 1."""
    dense_n = min(4 << 20, m + (300_000 if m < 16384 else 100_000))
    out = [("a^n", np.full(dense_n, ord("a"), dtype=np.uint8), np.full(m, ord("a"), dtype=np.uint8))]
    ab = np.resize(np.frombuffer(b"ab", dtype=np.uint8), dense_n + 1)
    out.append(("(ab)^k", ab, ab[: 2 * (m // 2)].copy()))
    out.append(("b(ab)^k", ab, ab[1: 2 * (m // 2) + 2].copy()))
    out += adversarial_cases(m, rng, scale=min(6 * m, 2 << 20))
    # random four-letter text with copies at 0, at n - m and across tile seams
    n = min(4 << 20, max(8 * m, 1 << 19))
    text = rng.integers(65, 69, size=n, dtype=np.uint8)
    pat = text[n // 3: n // 3 + m].copy()
    at = [0]
    while True:                          # the next 16 or 32 KiB seam past the previous copy, straddled three ways
        step = 32768 if len(at) % 2 else 16384
        seam = ((at[-1] + 2 * m) // step + 1) * step
        o = seam - (m // 2, 1, m - 1)[len(at) % 3]
        if o + 2 * m > n:
            break
        at.append(o)
    at.append(n - m)
    for o in at:
        text[o:o + m] = pat
    out.append(("seams", text, pat))
    x = rng.integers(65, 69, size=m + 1, dtype=np.uint8)
    out.append(("m=n-1 end", x.copy(), x[1:].copy()))
    out.append(("m=n-1 start", x.copy(), x[:-1].copy()))
    out.append(("m=n", x[:m].copy(), x[:m].copy()))
    return out


@pytest.mark.parametrize("m", LONG_MS)
def test_long_patterns_dense_and_adversarial(bmx, oracle, dev, monkeypatch, m):  # noqa: F811
    rng = np.random.default_rng(m + 17)
    coops = (1, 0) if m == 1024 else (None,)
    for name, text, pat_arr in long_pattern_texts(rng, m):
        pat = pat_arr.tobytes()
        want = kmp(oracle, text, pat)
        if name == "a^n":
            assert np.array_equal(want, np.arange(text.size - pat_arr.size + 1))
        if name == "seams":
            assert want.size >= 3
        for mis in MISALIGN:
            td = to_dev(text, dev, misalign=mis)
            for dense in (1, None):
                for coop in coops:
                    set_knobs(monkeypatch, BMX_DENSE_LANES=dense, BMX_COOP_VERIFY=coop)
                    check(bmx, td, pat, want, "auto", (m, name, mis, dense, coop), first=dense is None)
            del td


# ---------------------------------------------------------------------------------------------------------------
# 3. The multi-pattern kernel at its eligibility limits (7 <= m <= 4096, K <= 64)
# ---------------------------------------------------------------------------------------------------------------
def check_multi(bmx, oracle, text: np.ndarray, pats, tag=()):
    """search_multi_device (caps 0, 1, half, full; aligned and odd offset) and search_multi against K KMP runs."""
    wants = [kmp(oracle, text, p) for p in pats]
    full = max(1, max(w.size for w in wants))
    for mis in MISALIGN:
        td = to_dev(text, torch.device("cuda:0"), misalign=mis)
        for cap in sorted({0, 1, max(full // 2, 1), full}):
            got = bmx.search_multi_device(td, pats, max_positions=cap)
            assert len(got) == len(pats)
            for k, ((count, pos), want) in enumerate(zip(got, wants)):
                assert count == want.size, (*tag, mis, cap, k, len(pats[k]), count, want.size)
                if cap == 0:
                    assert pos is None
                else:
                    assert np.array_equal(pos.cpu().numpy(), want[:cap]), (*tag, mis, cap, k, len(pats[k]))
        del td
    for k, (count, pos) in enumerate(bmx.search_multi(text, pats)):
        assert count == wants[k].size and np.array_equal(pos, wants[k]), (*tag, "host", k, len(pats[k]))
    return wants


@pytest.mark.parametrize("tile", [16384, 32768])
def test_multi_pattern_gram_edges_and_longest_patterns(bmx, oracle, dev, monkeypatch, tile):  # noqa: F811
    """m_min 7 (no second hash word), 8, 11, 12-15 (a partial third word), 16, each with a 4096-byte pattern in the
    same set (halo at its limit, the pattern blob beyond the 4 KiB that fits in shared memory).  A 32 KiB multi tile
    leaves room for one pipeline stage next to a 4096-byte halo, so plan_scan scans such sets in 16 KiB tiles."""
    set_knobs(monkeypatch, BMX_MULTI_TILE=tile)
    rng = np.random.default_rng(tile + 1)
    n = (3 << 20) + 333
    text = rng.integers(65, 69, size=n, dtype=np.uint8)
    for m_min in (7, 8, 11, 12, 13, 15, 16):
        lens = [m_min, m_min + 1, 33, 300, 1024, 4095, 4096]
        pats = []
        for i, m in enumerate(lens):
            o = int(rng.integers(0, n - m))
            p = text[o:o + m].copy()
            for s in (16384 * (i + 1) - m // 2, n - m - 3 * i, (2 << 20) + 32768 * i - 1):   # seams and the text's end
                text[s:s + m] = p
            pats.append(p.tobytes())
        pats.append(pats[0][:-1] + bytes([pats[0][-1] ^ 1]))           # shares all grams but the last byte
        check_multi(bmx, oracle, text, pats, ("gram-edges", tile, m_min))
    # m_max <= 1024: a real 32 KiB multi tile (and a blob that fits in shared memory)
    pats = [text[o:o + m].tobytes() for o, m in ((100, 7), (5000, 12), (70000, 200), (1 << 20, 1024))]
    check_multi(bmx, oracle, text, pats, ("m_max 1024", tile))


def test_multi_pattern_full_probe_chains(bmx, oracle, dev):  # noqa: F811
    """64 patterns whose 256 (pattern, residue) table entries share one hash (every q-gram of the first 15 bytes is
    the same), 64 patterns that share their first 12 bytes, and patterns that share one gram at different residues."""
    rng = np.random.default_rng(64)
    n = (2 << 20) + 17
    base = rng.integers(97, 101, size=n, dtype=np.uint8)
    head = b"a" * 15
    same = [head + bytes(rng.integers(97, 101, size=int(rng.integers(1, 40)), dtype=np.uint8)) for _ in range(64)]
    prefix = bytes(rng.integers(97, 101, size=12, dtype=np.uint8))
    shared12 = [prefix + bytes(rng.integers(97, 101, size=int(rng.integers(1, 60)), dtype=np.uint8)) for _ in range(64)]
    gram = b"GRAMgramGRAM"
    residues = [b"x" * r + gram + b"yz" * (r + 1) for r in range(8)]
    for name, pats in (("one hash", same), ("shared 12", shared12), ("residues", residues)):
        text = base.copy()
        text[(1 << 20):(1 << 20) + 5000] = ord("a")                    # a long run: every word probes the full chain
        for i, p in enumerate(pats):
            for s in (16384 * (i + 1) + i, n - 40 - len(p) - 3 * i, 600_000 + 997 * i):
                text[s:s + len(p)] = np.frombuffer(p, dtype=np.uint8)
        wants = check_multi(bmx, oracle, text, pats, (name,))
        assert sum(w.size > 0 for w in wants) >= len(pats) // 2


def test_multi_pattern_longer_than_text_and_truncated_end(bmx, oracle, dev):  # noqa: F811
    """An eligible set with a pattern longer than the text (m_min <= n < m_max), and texts that end in a proper prefix
    of one of the patterns: the candidate check's end-of-text guard and the split kernel's p + m <= n guard."""
    rng = np.random.default_rng(11)
    long_pat = rng.integers(97, 100, size=4096, dtype=np.uint8)
    for n in (3000, 4095, 100_000):
        text = rng.integers(97, 100, size=n, dtype=np.uint8)
        cut = min(n - 10, 4095)
        text[n - cut:] = long_pat[:cut]                                # the text ends in a proper prefix of long_pat
        pats = [long_pat.tobytes(), long_pat[:7].tobytes(), long_pat[:12].tobytes(), long_pat[:cut - 1].tobytes(),
                long_pat[:cut].tobytes(), text[:9].tobytes()]
        wants = check_multi(bmx, oracle, text, pats, ("truncated end", n))
        assert wants[0].size == 0
        assert wants[4].size >= 1 and wants[4][-1] == n - cut


def test_multi_pattern_dense_union_second_pass(bmx, oracle, dev, monkeypatch):  # noqa: F811
    """Every start matches: the union list outgrows its first allocation (2^20 entries for this text) and the scan
    runs a second time with room for all of it."""
    n = 3_000_000
    text = np.full(n, ord("a"), dtype=np.uint8)
    text[2_000_000] = ord("b")
    pats = [b"a" * 7, b"a" * 12, b"a" * 6 + b"b", b"a" * 40]
    for tile in (16384, 32768):
        set_knobs(monkeypatch, BMX_MULTI_TILE=tile)
        wants = check_multi(bmx, oracle, text, pats, ("dense", tile))
        assert wants[0].size > (1 << 21)


def test_multi_pattern_ineligible_sets(bmx, oracle, dev):  # noqa: F811
    """A 4097-byte pattern or a 65th pattern sends the set pattern by pattern, with the same answers."""
    rng = np.random.default_rng(4097)
    n = (1 << 20) + 5
    text = rng.integers(65, 69, size=n, dtype=np.uint8)
    p4097 = text[5000:5000 + 4097].tobytes()
    text[700_000:700_000 + 4097] = np.frombuffer(p4097, dtype=np.uint8)
    small = [text[o:o + m].tobytes() for o, m in ((10, 7), (999, 9), (77_777, 15), (300_000, 64))]
    check_multi(bmx, oracle, text, small + [p4097], ("4097",))
    rnd = random.Random(65)
    pats = [text[o:o + m].tobytes() for o, m in ((rnd.randrange(n - 40), rnd.randint(7, 30)) for _ in range(65))]
    check_multi(bmx, oracle, text, pats, ("K=65",))
    check_multi(bmx, oracle, text, pats[:64], ("K=64",))


# ---------------------------------------------------------------------------------------------------------------
# 4. Counts and ranks past 2^32
# ---------------------------------------------------------------------------------------------------------------
def test_counts_and_ranks_past_2_pow_32(bmx, dev):  # noqa: F811
    """A 4.3 GB text of one letter: every start matches, so the answer is closed form.  With 2^20 positions of room
    a rank truncated to 32 bits anywhere in scan -> block scan -> expand would put hits of rank >= 2^32 into the
    first slots; the count-only path and find-first carry their own counters and keys."""
    n = (1 << 32) + (1 << 21) + 77
    td = torch.full((n,), ord("a"), dtype=torch.uint8, device=dev)
    cap = 1 << 20
    head = torch.arange(cap, device=dev)
    try:
        for m in (1, 2, 7, 40):
            pat = b"a" * m
            variants = ["auto", "window"] + (["qgram"] if m >= 7 else []) + (["shiftand"] if m <= 32 else [])
            for variant in variants:
                count, pos, _ = bmx.search_device(td, pat, variant=variant)
                assert count == n - m + 1 and pos is None, (m, variant, "count-only", count)
                count, pos, _ = bmx.search_device(td, pat, max_positions=cap, variant=variant)
                assert count == n - m + 1 and torch.equal(pos, head), (m, variant, "capped")
        got = bmx.search_multi_device(td, [b"a" * 7, b"a" * 12], max_positions=1000)
        for (count, pos), m in zip(got, (7, 12)):
            assert count == n - m + 1 and torch.equal(pos, head[:1000]), ("multi", m)
        # a zero text with one occurrence past 2^32 and one across the 2^32 boundary
        td.zero_()
        pat = b"needle\x01\x02\x03past32"
        m = len(pat)
        p = torch.frombuffer(bytearray(pat), dtype=torch.uint8).to(dev)
        want = [(1 << 32) + 5 - m, (1 << 32) + 5]                     # across the boundary, and right behind it
        for at in want:
            td[at:at + m] = p
        assert bmx.find_first_device(td, pat) == want[0]
        for variant in ("auto", "window", "qgram", "shiftand"):
            count, pos, _ = bmx.search_device(td, pat, max_positions=16, variant=variant)
            assert count == 2 and pos.cpu().tolist() == want, variant
        td[want[0]:want[0] + m] = 0
        assert bmx.find_first_device(td, pat) == want[1]
        count, pos, _ = bmx.search_device(td, pat, max_positions=16)
        assert count == 1 and pos.cpu().tolist() == want[1:]
    finally:
        del td
        torch.cuda.empty_cache()
