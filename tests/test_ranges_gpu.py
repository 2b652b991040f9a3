"""Many ranges of one text in one pass (bmx_search_ranges / bmx_search_ranges_device, host.search_ranges[_device]).

The contract: range d = [begin[d], end[d]) gets exactly what an ordinary search of text[begin[d]:end[d]] gets --
its count, and its positions relative to begin[d] at pos[offsets[d]:offsets[d+1]] -- so every case compares each
range with the oracle run on that range's slice.  The large cases derive the per-range truth from the oracle's
whole-text list with np.searchsorted and check a random sample of ranges slice by slice as well.
The argument checks at the top need no GPU; everything else is marked gpu."""
from __future__ import annotations

import ctypes
import random

import numpy as np
import pytest

from test_parity_gpu import dev, to_dev  # noqa: F401  (dev is a fixture)

GIB = 1 << 30


# ---------------------------------------------------------------------------------------------------------------
# CPU: argument checks and exports (no device is touched)
# ---------------------------------------------------------------------------------------------------------------
def _i64(*v):
    return (ctypes.c_int64 * max(len(v), 1))(*v)


def test_ranges_symbols_are_exported(bmx):
    lib = bmx._lib.load()
    for name in ("bmx_search_ranges", "bmx_search_ranges_device"):
        assert name in bmx._lib.EXPORTS and hasattr(lib, name)


def test_ranges_bad_arguments_are_rejected_without_touching_a_gpu(bmx):
    lib = bmx._lib.load()
    E = bmx._lib.BMX_E_BADARG
    text, n = b"abcabcabc", 9
    counts = (ctypes.c_uint64 * 4)()
    offs = _i64(0, 0, 0, 0, 0)
    pos = _i64(*[0] * 16)

    def host(begin, end, nr=None, pat=b"abc", m=3, pos_out=pos, cap=16, cnt=counts, off=offs, t=text, tn=n):
        nr = len(begin) if nr is None else nr
        return lib.bmx_search_ranges(0, t, tn, nr, _i64(*begin), _i64(*end), pat, m, pos_out, cap, cnt, off)

    assert host([0, 5], [3, 4]) == E                       # begin > end
    assert b"range 1" in lib.bmx_last_error()              # the bad range is named
    assert host([0, 2], [3, n + 1]) == E                   # end > n
    assert b"range 1" in lib.bmx_last_error()
    assert host([-1], [3]) == E                            # negative begin
    assert b"range 0" in lib.bmx_last_error()
    assert host([0], [3], nr=-1) == E                      # nranges < 0
    assert host([0], [3], cap=-1) == E                     # pos_cap < 0
    assert host([0], [3], pat=None) == E
    assert host([0], [3], m=0) == E                        # empty pattern
    assert host([0], [3], cnt=None) == E
    assert host([0], [3], off=None) == E
    assert host([0], [3], t=None) == E                     # NULL text with n > 0
    assert host([0], [3], tn=-1) == E
    assert lib.bmx_search_ranges(0, text, n, 1, None, _i64(3), b"abc", 3, pos, 16, counts, offs) == E
    assert lib.bmx_search_ranges(0, text, n, 1, _i64(0), None, b"abc", 3, pos, 16, counts, offs) == E

    total = ctypes.c_uint64()
    fake = ctypes.c_void_p(0x1000)   # never dereferenced: every check below fails before any device work

    def device(nr=1, b=fake, e=fake, pat=b"abc", m=3, cap=16, cnt=fake, off=fake, tot=ctypes.byref(total), t=fake, tn=n):
        return lib.bmx_search_ranges_device(t, tn, nr, b, e, pat, m, fake, cap, cnt, off, tot, None)

    assert device(nr=-1) == E
    assert device(cap=-1) == E
    assert device(b=None) == E
    assert device(e=None) == E
    assert device(cnt=None) == E
    assert device(off=None) == E
    assert device(tot=None) == E
    assert device(pat=None) == E
    assert device(m=0) == E
    assert device(t=None) == E
    assert device(tn=-1) == E


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


def _torch():
    return pytest.importorskip("torch")


def find_all(text: bytes, pat: bytes) -> np.ndarray:
    """All (overlapping) occurrences with bytes.find: for patterns too long for the oracle's O(m^3) tables."""
    out, i = [], text.find(pat)
    while i >= 0:
        out.append(i)
        i = text.find(pat, i + 1)
    return np.array(out, dtype=np.int64)


def slice_truth(oracle, text: bytes, pat: bytes, begin, end):
    """(counts, offsets, positions): one ordinary oracle search per range slice."""
    lists = []
    for b, e in zip(begin, end):
        piece = text[int(b): int(e)]
        if len(piece) < len(pat):
            lists.append(np.zeros(0, dtype=np.int64))
        else:
            lists.append(oracle.search(piece, pat) if len(pat) <= 64 else find_all(piece, pat))
    counts = np.array([x.size for x in lists], dtype=np.uint64)
    offsets = np.concatenate([[0], np.cumsum(counts, dtype=np.int64)]).astype(np.int64)
    pos = np.concatenate(lists) if lists else np.zeros(0, dtype=np.int64)
    return counts, offsets, pos.astype(np.int64)


def list_truth(whole: np.ndarray, m: int, begin, end):
    """(counts, offsets, positions) from the whole text's ascending match list."""
    begin = np.asarray(begin, dtype=np.int64)
    end = np.asarray(end, dtype=np.int64)
    a = np.searchsorted(whole, begin, side="left")
    b = np.searchsorted(whole, end - m + 1, side="left")
    counts = np.where(end - begin >= m, b - a, 0).astype(np.int64)
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    total = int(offsets[-1])
    idx = np.arange(total, dtype=np.int64) - np.repeat(offsets[:-1], counts) + np.repeat(a, counts)
    pos = whole[idx] - np.repeat(begin, counts)
    return counts.astype(np.uint64), offsets, pos


def run_host(bmx, text, pat, begin, end, **kw):
    c, o, p = bmx.search_ranges(text, pat, np.asarray(begin, dtype=np.int64), np.asarray(end, dtype=np.int64), **kw)
    return c, o, p


def run_device(bmx, td, pat, begin, end, dev, **kw):
    torch = _torch()
    bd = torch.as_tensor(np.asarray(begin, dtype=np.int64), device=dev)
    ed = torch.as_tensor(np.asarray(end, dtype=np.int64), device=dev)
    c, o, p = bmx.search_ranges_device(td, pat, bd, ed, **kw)
    return c.cpu().numpy().astype(np.uint64), o.cpu().numpy(), (None if p is None else p.cpu().numpy())


def assert_same(got, want, tag, cap=None):
    c, o, p = got
    wc, wo, wp = want
    assert np.array_equal(c, wc), (tag, "counts")
    assert np.array_equal(o, wo), (tag, "offsets")
    wp = wp if cap is None else wp[:cap]
    assert p is not None and np.array_equal(p, wp), (tag, "positions", None if p is None else p.size, wp.size)


def check_both(bmx, dev, text: bytes, pat: bytes, begin, end, want, tag, misalign=0):
    """Host entry (room for all, a cap inside the list, counts only) and device entry against `want`."""
    total = int(want[1][-1])
    assert_same(run_host(bmx, text, pat, begin, end), want, (tag, "host"))
    cap = max(total // 2, 1)
    assert_same(run_host(bmx, text, pat, begin, end, max_positions=cap), want, (tag, "host cap"), cap=cap)
    c, o, p = run_host(bmx, text, pat, begin, end, max_positions=0)
    assert np.array_equal(c, want[0]) and np.array_equal(o, want[1]) and p.size == 0, (tag, "host counts only")
    td = to_dev(text, dev, misalign)
    assert_same(run_device(bmx, td, pat, begin, end, dev, max_positions=max(total, 1)), want, (tag, "device"))
    c, o, p = run_device(bmx, td, pat, begin, end, dev)
    assert np.array_equal(c, want[0]) and np.array_equal(o, want[1]) and p is None, (tag, "device counts only")


def random_text(n: int, seed: int, alphabet: bytes = b"abcd") -> bytes:
    rnd = np.random.default_rng(seed)
    return np.frombuffer(alphabet, dtype=np.uint8)[rnd.integers(0, len(alphabet), n)].tobytes()


def plant(text: bytes, pat: bytes, where) -> bytes:
    buf = bytearray(text)
    for w in where:
        w = int(w)
        if 0 <= w and w + len(pat) <= len(buf):
            buf[w: w + len(pat)] = pat
    return bytes(buf)


@gpu
def test_tiling_ranges_never_count_a_match_across_a_seam(bmx, oracle, dev):
    n, m = 300_000, 8
    pat = b"abcdabcd"
    rnd = random.Random(1)
    seams = sorted(32 * s for s in rnd.sample(range(1, n // 32 - 1), 400))   # seams at least 4 m apart
    text = random_text(n, 1, b"abcd")
    text = plant(text, pat, [rnd.randrange(0, n - m) for _ in range(300)])
    text = plant(text, pat, [s - m // 2 for s in seams])            # one match across every seam, planted last
    begin = [0] + seams
    end = seams + [n]
    want = slice_truth(oracle, text, pat, begin, end)
    check_both(bmx, dev, text, pat, begin, end, want, "tiling")
    whole = oracle.search(text, pat)
    seam = np.asarray(seams, dtype=np.int64)
    nxt = np.searchsorted(seam, whole, side="right")                 # first seam behind each match start
    straddle = (nxt < seam.size) & (seam[np.minimum(nxt, seam.size - 1)] < whole + m)
    assert int(straddle.sum()) >= len(seams) and int(want[1][-1]) == whole.size - int(straddle.sum())


@gpu
def test_edge_ranges(bmx, oracle, dev):
    n, pat = 100_000, b"abca"
    text = plant(random_text(n, 2), pat, range(0, n, 997))
    begin = [0, 5, 10, 10, n, n - 3, 500, 400, 400, 400, 300, 77_000, 0, 123]
    end = [0, 5, 13, 14, n, n, 900, 1200, 1200, 1200, 50_000, 70_000 + 7_005, n, 123 + 4]
    want = slice_truth(oracle, text, pat, begin, end)
    check_both(bmx, dev, text, pat, begin, end, want, "edges", misalign=3)
    # one range equal to the whole text is bmx.search exactly
    count, pos = bmx.search(text, pat)
    c, o, p = run_host(bmx, text, pat, [0], [n])
    assert int(c[0]) == count and int(o[1]) == count and np.array_equal(p, pos)
    c, o, p = run_device(bmx, to_dev(text, dev), pat, [0], [n], dev, max_positions=count)
    assert int(c[0]) == count and np.array_equal(p, pos)
    # no ranges at all, and ranges of a text shorter than the pattern
    c, o, p = run_host(bmx, text, pat, [], [])
    assert c.size == 0 and list(o) == [0] and p.size == 0
    c, o, p = run_device(bmx, to_dev(text, dev), pat, [], [], dev, max_positions=4)
    assert c.size == 0 and list(o) == [0] and p.size == 0
    c, o, p = run_device(bmx, to_dev(b"abc", dev), pat, [0, 1], [3, 3], dev, max_positions=4)
    assert list(c) == [0, 0] and list(o) == [0, 0, 0] and p.size == 0


@gpu
def test_ranges_in_the_middle_of_a_large_text(bmx, oracle, dev):
    torch = _torch()
    n, m = 64 << 20, 12
    alpha = bmx.synth.ALPHABETS["dna"]
    t = torch.empty(n, dtype=torch.uint8, device=dev)
    bmx.synth.fill_device(t, 0, 71, alpha)
    pat = bmx.synth.pattern_from_stream(m, 71, alpha)
    mid = n // 2
    bmx.synth.plant_device(t, pat, bmx.synth.plant_offsets(1 << 20, m, 2000, 71, lo=mid))
    text = t.cpu().numpy().tobytes()
    rnd = random.Random(3)
    begin = [mid + rnd.randrange(0, 1 << 20) for _ in range(200)]
    end = [b + rnd.randrange(0, 20_000) for b in begin]
    want = slice_truth(oracle, text, pat, begin, end)
    assert int(want[1][-1]) > 50
    assert_same(run_host(bmx, text, pat, begin, end), want, "middle host")
    assert_same(run_device(bmx, t, pat, begin, end, dev, max_positions=int(want[1][-1])), want, "middle device")


@gpu
@pytest.mark.parametrize("m, alphabet", [(1, b"abcdefgh"), (2, b"abcd"), (3, b"abcd"), (4, b"abcd"), (5, b"ACGT"),
                                         (7, b"abcd"), (16, b"abc"), (1024, b"ab"), (1500, b"ab")])
def test_every_filter_kind(bmx, oracle, dev, m, alphabet):
    n = 400_000
    text = random_text(n, 10 + m, alphabet)
    pat = text[1000: 1000 + m]
    rnd = random.Random(m)
    text = plant(text, pat, [rnd.randrange(0, n - m) for _ in range(200)])
    begin = [rnd.randrange(0, n) for _ in range(150)]
    end = [min(n, b + rnd.choice([0, m - 1, m, m + 1, 3000, 40_000])) for b in begin]
    want = slice_truth(oracle, text, pat, begin, end)
    assert int(want[1][-1]) > 0
    check_both(bmx, dev, text, pat, begin, end, want, ("m", m), misalign=m % 7)


@gpu
def test_dense_list_grows_and_caps_cut_anywhere(bmx, dev):
    """8 MiB of 'a' with 'aaa': 8 Mi hits against a first guess of 1 Mi, so L grows on a second pass."""
    torch = _torch()
    n = 8 << 20
    begin = np.array([100, 0, 5 << 20, 3 << 20, 7], dtype=np.int64)
    end = np.array([200_100, 2, n, (3 << 20) + 1000, 7 + 3], dtype=np.int64)
    counts = np.maximum(end - begin - 2, 0)
    offsets = np.concatenate([[0], np.cumsum(counts)])
    pos = np.concatenate([np.arange(c, dtype=np.int64) for c in counts])
    want = (counts.astype(np.uint64), offsets, pos)
    text = b"a" * n
    td = torch.full((n,), ord("a"), dtype=torch.uint8, device=dev)
    for cap in (None, int(offsets[1]) + 17, int(offsets[3]), 0):   # all, inside a range, at a range edge, none
        bmx._lib.load().bmx_release_memory(-1)                    # the position buffer starts from its first guess
        assert_same(run_host(bmx, text, b"aaa", begin, end, max_positions=cap), want, ("host", cap), cap=cap)
        bmx._lib.load().bmx_release_memory(-1)
        got = run_device(bmx, td, b"aaa", begin, end, dev, max_positions=int(offsets[-1]) if cap is None else cap)
        if cap == 0:
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], offsets) and got[2] is None
        else:
            assert_same(got, want, ("device", cap), cap=cap)
    assert_same(run_device(bmx, td, b"aaa", begin, end, dev, max_positions=int(offsets[-1])), want, "device all")


@gpu
def test_gather_balance_one_giant_range_and_a_million_tiny_ones(bmx, oracle, dev):
    torch = _torch()
    half = 16 << 20
    host = np.empty(2 * half, dtype=np.uint8)
    host[:half] = ord("A")
    host[half:] = bmx.synth.fill_host(0, half, 5, b"ACGT")
    pat = b"AAAA"
    whole = oracle.search_np(host, pat)
    rnd = np.random.default_rng(7)
    tiny_b = rnd.integers(half, 2 * half - 64, 1_000_000)
    tiny_e = tiny_b + rnd.integers(0, 65, tiny_b.size)
    begin = np.concatenate([[0], tiny_b[:500_000], [17], tiny_b[500_000:]]).astype(np.int64)
    end = np.concatenate([[half + 2], tiny_e[:500_000], [17 + 4], tiny_e[500_000:]]).astype(np.int64)
    want = list_truth(whole, len(pat), begin, end)
    assert int(want[0][0]) >= half - 3 and int(want[1][-1]) > half
    td = torch.from_numpy(host).to(dev)
    got = run_device(bmx, td, pat, begin, end, dev, max_positions=int(want[1][-1]))
    assert_same(got, want, "balance device")
    assert_same(run_host(bmx, host, pat, begin, end), want, "balance host")
    text = host.tobytes()
    for d in rnd.choice(begin.size, 200, replace=False):
        c, o, p = slice_truth(oracle, text, pat, [begin[d]], [end[d]])
        assert int(got[0][d]) == int(c[0]) and np.array_equal(got[2][got[1][d]: got[1][d + 1]], p), d
    # a ragged batch of a million tiny documents: begin = offsets[:-1], end = offsets[1:]
    cuts = np.sort(rnd.integers(0, host.size, 1_000_000 - 1))
    doc = np.concatenate([[0], cuts, [host.size]]).astype(np.int64)
    want = list_truth(whole, len(pat), doc[:-1], doc[1:])
    dd = torch.as_tensor(doc, device=dev)
    c, o, p = bmx.search_ranges_device(td, pat, dd[:-1], dd[1:], max_positions=int(want[1][-1]))
    assert np.array_equal(c.cpu().numpy().astype(np.uint64), want[0]) and np.array_equal(o.cpu().numpy(), want[1])
    assert np.array_equal(p.cpu().numpy(), want[2])


@gpu
@pytest.mark.parametrize("knobs", [{"BMX_H2D_CHUNK_KB": "64"}, {"BMX_RESIDENT_MAX_MB": "0", "BMX_H2D_CHUNK_KB": "64"}])
def test_host_entry_chunked_and_ring(bmx, oracle, dev, monkeypatch, knobs):
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    n, m = 3 << 20, 9
    chunk = 64 << 10
    pat = b"abcabcabd"
    rnd = random.Random(9)
    text = random_text(n, 9, b"abcd")
    text = plant(text, pat, [k * chunk - rnd.randrange(1, m) for k in range(1, n // chunk)])   # matches across chunk seams
    text = plant(text, pat, [rnd.randrange(0, n - m) for _ in range(500)])
    begin = [k * chunk - rnd.randrange(0, 3000) for k in range(1, n // chunk)] + [rnd.randrange(0, n) for _ in range(100)]
    end = [min(n, b + rnd.randrange(0, 200_000)) for b in begin]
    want = slice_truth(oracle, text, pat, begin, end)
    assert int(want[1][-1]) > 100
    assert_same(run_host(bmx, text, pat, begin, end), want, ("host", knobs))
    assert_same(run_host(bmx, text, pat, begin, end, max_positions=37), want, ("host cap", knobs), cap=37)


@gpu
def test_device_entry_misaligned_view_and_a_bad_range(bmx, oracle, dev):
    torch = _torch()
    n, pat = 200_000, b"dcba"
    text = plant(random_text(n, 4), pat, range(3, n, 1231))
    begin = [0, 1000, 50_000, 7]
    end = [n, 90_000, 50_003, 7]
    want = slice_truth(oracle, text, pat, begin, end)
    for k in (1, 5, 13):
        td = to_dev(text, dev, misalign=k)
        assert_same(run_device(bmx, td, pat, begin, end, dev, max_positions=int(want[1][-1])), want, ("misalign", k))
    td = to_dev(text, dev, misalign=5)
    for bad_b, bad_e in [(0, n + 1), (10, 9), (-4, 5), (n + 1, n + 2)]:
        bd = torch.tensor(begin + [bad_b], dtype=torch.int64, device=dev)
        ed = torch.tensor(end + [bad_e], dtype=torch.int64, device=dev)
        with pytest.raises(bmx.BmxError) as e:
            bmx.search_ranges_device(td, pat, bd, ed, max_positions=100)
        assert e.value.code == bmx._lib.BMX_E_BADARG and "range 4" in str(e.value)
        assert_same(run_device(bmx, td, pat, begin, end, dev, max_positions=int(want[1][-1])), want, ("after", bad_b))


@gpu
def test_text_past_4GiB_with_ranges_across_2_to_32(bmx, oracle, dev):
    torch = _torch()
    n, m, seed = 4 * GIB + (64 << 20), 16, 81
    alpha = bmx.synth.ALPHABETS["ascii95"]
    t = torch.empty(n, dtype=torch.uint8, device=dev)
    bmx.synth.fill_device(t, 0, seed, alpha)
    pat = bmx.synth.pattern_from_stream(m, seed, alpha)
    edge = 1 << 32
    plants = [edge - 8, edge + 100, edge - 3000, edge + 70_000, 17, n - m]   # edge - 8 straddles 2^32
    bmx.synth.plant_device(t, pat, plants)
    begin = [edge - 1000, edge - 5, edge - m + 3, edge - 20_000, 0, n - 100_000, edge, edge - 3000]
    end = [edge + 1000, edge + 5, edge + m, edge + 100_000, 1000, n, edge + m + 5, edge - 3000 + m]
    lists = []
    for b, e in zip(begin, end):
        lists.append(oracle.search(t[b:e].cpu().numpy().tobytes(), pat))
    counts = np.array([x.size for x in lists], dtype=np.uint64)
    want = (counts, np.concatenate([[0], np.cumsum(counts, dtype=np.int64)]), np.concatenate(lists))
    assert int(counts[2]) >= 1 and int(counts[3]) >= 4 and int(counts[7]) >= 1
    assert_same(run_device(bmx, t, pat, begin, end, dev, max_positions=int(counts.sum())), want, "past 2^32")
    del t
    torch.cuda.empty_cache()


@gpu
@pytest.mark.parametrize("nparts", [1000, 10_000])
def test_partition_mirror_on_the_english_fixture(bmx, oracle, golden, nparts):
    text = golden.text("input5L")
    se = bmx.partition_words(text, nparts)
    for pat in (b"is", b"the", b"e", b"position", b" "):
        assert np.array_equal(bmx.search_partitions(text, pat, se), oracle.search_partitions(text, pat, se)), (pat, nparts)
    # the same ranges through search_ranges, with positions
    begin = se[0::2].astype(np.int64)
    end = np.maximum(se[1::2].astype(np.int64) + 1, begin)
    want = slice_truth(oracle, text, b"is", begin, end)
    assert_same(run_host(bmx, text, b"is", begin, end), want, ("english", nparts))
