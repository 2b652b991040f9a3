"""Ordered emission at the exact boundaries between its code paths, with guard bands around every output buffer.

bmx.h promises that at most pos_cap positions are written, the smallest ones, and nothing else.  Every test here
passes an output pointer into a larger allocation filled with a sentinel, G entries behind the start (16-byte
aligned) or G + 1 entries (out[0] only 8-byte aligned), and checks that the first min(count, cap) entries equal the
KMP matcher's list (oracle_kmp_search, no Boyer-Moore logic) and that every other entry -- in front, between count
and cap, at cap and behind -- still holds the sentinel.  The calls go through ctypes directly, because the host.py
wrappers allocate exact-size buffers and pass NULL for a cap of 0.

The texts are built from hit sets in "V space", where the expand kernel decides which path a hit takes: start p of
a text at address A belongs to segment u // 2048 (item u // 32768, block u // 2 MiB) with u = p + (A & 15) -
owner_offset, owner_offset being -3 for QGRAM and the multi-pattern kernel and 0 otherwise.  A hit set becomes a
text of 'b' with runs of 'a' searched for 'a' * m.  Each case asserts the intended shape on the KMP list before it
runs, so a shape that missed its path threshold fails loudly instead of testing nothing.  The caps come from the
truth's ranks: the first and end rank of every segment, item and block that holds hits, each +-1."""
from __future__ import annotations

import ctypes
from ctypes import byref, c_int64, c_uint64, c_void_p

import numpy as np
import pytest

from test_exact_reference import kmp
from test_parity_gpu import dev, to_dev  # noqa: F401  (dev is a fixture)

torch = pytest.importorskip("torch")

SEG, ITEM_SEGS, BLOCK_SEGS = 2048, 16, 1024
ITEM, BLOCK = SEG * ITEM_SEGS, SEG * BLOCK_SEGS
SOLO_MAX, STAGE, FLAT_MAX, SPARSE_SEGS, DENSE_BLOCK = 64, 96, 1024, 3, 1 << 17   # bmx_scan.cu, bmx_internal.h
SENT = 0x5A5A5A5A5A5A5A5A
G = 32                                          # guard entries on each side
OFFSETS = (G, G + 1)                            # out[0] 16-byte aligned, out[0] 8-byte aligned only
LEADS = (0, 5, 15)
BASES = (0, (1 << 40) + 7)
VARIANT_IDS = {"qgram": 1, "window": 2, "shiftand": 3}
# (label, variant, m): exact filters of one and three bytes, Shift-And, QGRAM (owner offset -3), a verifying WINDOW
VARIANTS = [("window-m1", "window", 1), ("window-m3", "window", 3), ("shiftand-m1", "shiftand", 1),
            ("qgram-m7", "qgram", 7), ("window-m16", "window", 16)]


def owner_of(variant: str) -> int:
    return -3 if variant == "qgram" else 0


# ---------------------------------------------------------------------------------------------------------------
# Shape builder (CPU)
# ---------------------------------------------------------------------------------------------------------------
SEG_COUNTS = (1, 63, 64, 65, 95, 96, 97, 2047, 2048)
# one work item each (segment index inside the item -> hits), every other item of block 0 stays empty
ITEM_SHAPES = [(f"segment-{h}", {1: h}) for h in SEG_COUNTS] + [
    ("sparse-3segs-96", {1: 32, 5: 32, 9: 32}),              # the most the sparse path takes
    ("flat-4segs-96", {1: 24, 5: 24, 9: 24, 13: 24}),         # one segment too many for it
    ("flat-3segs-97", {1: 32, 5: 32, 9: 33}),                 # one hit too many for it
    ("flat-1024", {s: 64 for s in range(16)}),                # the most the flat path takes
    ("segments-1025", {**{s: 64 for s in range(15)}, 15: 65}),
    ("segments-mixed", {1: 64, 3: 65, 5: 96, 7: 2048}),       # solo, warp, staged and full segments in one item
]
TEXT_N = 5 * BLOCK + 150_077                    # blocks 0-4 and a partial block 5


def seg_hits(s: int, h: int, m: int) -> np.ndarray:
    """h hits in V-space segment s: spread over all lanes and slabs when runs of 'a' stay m + 1 apart, else one run."""
    u0 = s * SEG
    stride = SEG // h
    if h < SEG and stride >= m + 1:
        return u0 + stride * np.arange(h, dtype=np.int64)
    a = (SEG - h) // 2
    return np.arange(u0 + a, u0 + a + h, dtype=np.int64)


def dense_block(b: int, total: int) -> dict:
    """Segment -> hits for block b: one segment of every class (every other segment, so runs stay apart), a
    remainder segment and full segments up to `total`."""
    segs = {b * BLOCK_SEGS + 1 + 2 * i: h for i, h in enumerate(SEG_COUNTS)}
    rest = total - sum(SEG_COUNTS)
    full, rem = divmod(rest, SEG)
    first_full = b * BLOCK_SEGS + 2 * len(SEG_COUNTS) + 3
    segs[first_full - 2] = rem
    segs.update({first_full + i: SEG for i in range(full)})
    return segs


def layout(m: int, lead: int, owner: int):
    """(hits in V space, named shape checks) for the shapes text of TEXT_N bytes.
    Block 0: ITEM_SHAPES in items 3, 5, 7, ...; block 1: 2^17 - 1 hits (sparse, the last sum below the dense switch);
    block 2: 2^17 hits (dense: ticket-ordered phase 2); blocks 3-4: hits on the first and last start of a segment,
    an item and a block; the first and the last start of the text; a dense final partial block."""
    d = lead - owner                                  # u of text position 0
    segs, checks = {}, []
    for i, (name, spec) in enumerate(ITEM_SHAPES):
        item = 2 * i + 3
        segs.update({item * ITEM_SEGS + s: h for s, h in spec.items()})
        checks.append((name, "item", item, sum(spec.values()), len(spec)))
    for b, total in ((1, DENSE_BLOCK - 1), (2, DENSE_BLOCK)):
        segs.update(dense_block(b, total))
        checks.append((f"block-{total}", "block", b, total, None))
    hits = [seg_hits(s, h, m) for s, h in segs.items()]
    S, I, J = 3 * BLOCK + 10 * ITEM + 7 * SEG, 3 * BLOCK + 20 * ITEM, 3 * BLOCK + 30 * ITEM
    edges = [d,                                       # first start of the text
             S, S + SEG - 1,                          # first and last start of one segment
             I, I + ITEM - 1,                         # first and last start of one item
             J - 1, J,                                # last start of an item, first of the next
             4 * BLOCK - 1, 4 * BLOCK, 5 * BLOCK - 1]  # last start of block 3, first and last of block 4
    last = TEXT_N - m + d                             # last start of the text ends the dense run of block 5
    hits += [np.array(edges, dtype=np.int64), np.arange(5 * BLOCK + 8000, last + 1, dtype=np.int64)]
    checks.append(("partial-dense", "partial", 5, DENSE_BLOCK, None))
    return np.unique(np.concatenate(hits)), checks


def realize(hits_u: np.ndarray, m: int, lead: int, owner: int, n: int) -> tuple[np.ndarray, np.ndarray]:
    """Text positions and the text whose occurrences of 'a' * m are exactly those hits."""
    p = hits_u - lead + owner
    assert p.size and p[0] >= 0 and p[-1] <= n - m, "hit outside the text"
    gaps = np.diff(p)
    assert np.all((gaps == 1) | (gaps >= m + 1)), "runs of 'a' closer than m + 1: they would merge into more hits"
    text = np.full(n, ord("b"), dtype=np.uint8)
    for j in range(m):
        text[p + j] = ord("a")
    return p, text


def profile(truth: np.ndarray, lead: int, owner: int, tile: int, n: int):
    """Per-segment counts, per-item totals and per-block sums of a hit list, as the scan kernel's tiles lay them out:
    the last block covers whole tiles, num_segs = tiles * tile / 2048."""
    u = truth + lead - owner
    tiles = -(-(lead + n) // tile)
    num_segs = tiles * (tile // SEG)
    num_blocks = -(-num_segs // BLOCK_SEGS)
    seg = np.bincount(u // SEG, minlength=num_segs)
    assert seg.size == num_segs
    item = np.bincount(u // ITEM, minlength=num_blocks * (BLOCK_SEGS // ITEM_SEGS))
    block = np.bincount(u // BLOCK, minlength=num_blocks)
    return seg, item, block


def assert_shapes(truth, checks, lead, owner, tile, n):
    seg, item, block = profile(truth, lead, owner, tile, n)
    for name, kind, idx, total, nsegs in checks:
        if kind == "item":
            segs = seg[idx * ITEM_SEGS:(idx + 1) * ITEM_SEGS]
            assert item[idx] == total and np.count_nonzero(segs) == nsegs, (name, item[idx], segs)
            assert item[idx - 1] == 0 and item[idx + 1] == 0, (name, "neighbours")
            if name == "sparse-3segs-96":
                assert total <= STAGE and nsegs <= SPARSE_SEGS
            elif name.startswith("flat-"):
                assert total <= FLAT_MAX and not (total <= STAGE and nsegs <= SPARSE_SEGS)
            elif name.startswith("segments-"):
                assert total > FLAT_MAX
        elif kind == "block":
            assert block[idx] == total, (name, block[idx])
            classes = seg[idx * BLOCK_SEGS:(idx + 1) * BLOCK_SEGS]
            for lo, hi in ((1, SOLO_MAX), (SOLO_MAX + 1, STAGE - 1), (STAGE, SEG - 1), (SEG, SEG)):
                assert np.any((classes >= lo) & (classes <= hi)), (name, lo, hi)
        else:                                           # the last block is partial and dense
            assert block.size == idx + 1 and block[idx] >= total and seg.size % BLOCK_SEGS != 0, (name, block)
    assert block[1] < DENSE_BLOCK <= block[2]


def rank_caps(truth, lead, owner, tile, n, first_block=0):
    """Caps r0, r0+1, r1-1, r1, r1+1 of every segment, item and block with hits (of full segments only those at the
    ends of a run), plus 0, 1, C-1, C and C+1; units in front of block `first_block` are left out."""
    seg, item, block = profile(truth, lead, owner, tile, n)
    inner_full = (seg == SEG) & (np.roll(seg, 1) == SEG) & (np.roll(seg, -1) == SEG)
    C = truth.size
    caps = {0, 1, C - 1, C, C + 1}
    for counts, pick, per_block in ((seg, (seg > 0) & ~inner_full, BLOCK_SEGS),
                                    (item, item > 0, BLOCK_SEGS // ITEM_SEGS), (block, block > 0, 1)):
        pick[:first_block * per_block] = False
        ends = np.cumsum(counts)
        starts = ends - counts
        for r0, r1 in zip(starts[pick], ends[pick]):
            caps.update((int(r0), int(r0) + 1, int(r1) - 1, int(r1), int(r1) + 1))
    return sorted(c for c in caps if c >= 0)


def shapes_text(oracle, variant: str, m: int, lead: int):
    owner = owner_of(variant)
    hits_u, checks = layout(m, lead, owner)
    p, text = realize(hits_u, m, lead, owner, TEXT_N)
    truth = kmp(oracle, text, b"a" * m)
    assert np.array_equal(truth, p), "the text holds other hits than the ones it was built from"
    return text, truth, checks


@pytest.mark.parametrize("lead", LEADS)
def test_shape_builder_reaches_every_threshold(oracle, lead):
    """CPU: every shape, for every lead and owner offset, is a text whose KMP list is the intended hit set, and the
    per-segment, per-item and per-block profile of that list sits exactly at the thresholds it is meant to hit."""
    for _label, variant, m in VARIANTS:
        text, truth, checks = shapes_text(oracle, variant, m, lead)
        for tile in (16384, 32768):
            assert_shapes(truth, checks, lead, owner_of(variant), tile, text.size)
        caps = rank_caps(truth, lead, owner_of(variant), 32768, text.size)
        assert caps[0] == 0 and caps[-1] == truth.size + 1


# ---------------------------------------------------------------------------------------------------------------
# Guarded device buffers
# ---------------------------------------------------------------------------------------------------------------
def lib_of(bmx):
    return bmx._lib.load()


def ok(bmx, rc):
    bmx._lib.check(rc)


def stream_ptr():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def guarded(size: int, device="cuda:0"):
    return torch.full((size,), SENT, dtype=torch.int64, device=device)


def expect(size: int, spans):
    """Sentinel everywhere except the (offset, values) spans."""
    e = np.full(size, SENT, dtype=np.int64)
    for off, vals in spans:
        e[off:off + len(vals)] = vals
    return e


def assert_same(got: np.ndarray, want: np.ndarray, tag):
    if not np.array_equal(got, want):
        bad = np.flatnonzero(got != want)
        i = int(bad[0])
        raise AssertionError(f"{tag}: {bad.size} entries differ, first at buffer index {i}: "
                             f"got {int(got[i]):#x}, want {int(want[i]):#x}")


def check_device_caps(bmx, td, pat: bytes, variant: str, base: int, truth: np.ndarray, caps, off: int, tag):
    """bmx_search_device_ex into a guarded buffer for every cap: exact count, exact prefix, sentinel elsewhere."""
    lib = lib_of(bmx)
    want = torch.from_numpy(truth + base).to(td.device)
    C = truth.size
    for cap in caps:
        k = min(C, cap)
        buf = guarded(off + cap + G, td.device)
        count = c_uint64()
        ok(bmx, lib.bmx_search_device_ex(c_void_p(td.data_ptr()), td.numel(), pat, len(pat), c_int64(base),
                                         c_void_p(buf.data_ptr() + 8 * off), cap, byref(count), VARIANT_IDS[variant],
                                         None, stream_ptr()))
        assert count.value == C, (*tag, cap, "count", count.value, C)
        exp = guarded(buf.numel(), td.device)
        exp[off:off + k] = want[:k]
        if not torch.equal(buf, exp):
            assert_same(buf.cpu().numpy(), exp.cpu().numpy(), (*tag, "cap", cap))


@pytest.mark.gpu
@pytest.mark.parametrize("label,variant,m", VARIANTS, ids=[v[0] for v in VARIANTS])
def test_device_emission_at_path_boundaries(bmx, oracle, dev, monkeypatch, label, variant, m):  # noqa: F811
    """Every shape, leads 0/5/15, pos_base 0 and 2^40 + 7 (the latter with out[0] off the 16-byte grid), every
    rank-derived cap; the end-of-text shapes also with 16 KiB tiles, and one pass with a one-CTA expand grid (four
    item flags per lane)."""
    pat = b"a" * m
    owner = owner_of(variant)
    for lead in LEADS:
        text, truth, checks = shapes_text(oracle, variant, m, lead)
        td = to_dev(text, dev, misalign=lead)
        assert td.data_ptr() % 16 == lead
        for tile in (32768, 16384):
            monkeypatch.setenv("BMX_TILE", str(tile))
            assert_shapes(truth, checks, lead, owner, tile, text.size)
            # 32 KiB tiles (the default): every shape; 16 KiB tiles: blocks 3 to 5 (text edges, partial dense block)
            caps = rank_caps(truth, lead, owner, tile, text.size, first_block=0 if tile == 32768 else 3)
            for base, off in zip(BASES, OFFSETS):
                if tile == 16384 and base:
                    continue
                check_device_caps(bmx, td, pat, variant, base, truth, caps, off, (label, lead, tile, base, off))
        if label == "window-m1" and lead == 5:
            monkeypatch.setenv("BMX_TILE", "32768")
            monkeypatch.setenv("BMX_EXPAND_GRID", "1")
            caps = rank_caps(truth, lead, owner, 32768, text.size)
            check_device_caps(bmx, td, pat, variant, BASES[1], truth, caps, OFFSETS[0], (label, lead, "grid1"))
            monkeypatch.delenv("BMX_EXPAND_GRID")
        del td


# ---------------------------------------------------------------------------------------------------------------
# Chains: the scanner API, the exported result, host ingest in chunks, the small-host read-back
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("label,variant,m", [VARIANTS[0], VARIANTS[3], VARIANTS[4]], ids=["window-m1", "qgram-m7", "window-m16"])
def test_scanner_chain_caps_at_every_carry(bmx, oracle, dev, label, variant, m):  # noqa: F811
    """One search as a chain of scans over pieces cut at segment and tile seams and at odd offsets (each piece has its
    own lead and its own pos_base): caps c_k - 1, c_k, c_k + 1 around the running count after every piece, where the
    expand kernel of the next scan ranks from the carried count.  Then bmx_scanner_export_result with head values
    0, 1, held - 1, held and held + 3 into a guarded destination."""
    lib = lib_of(bmx)
    pat = b"a" * m
    text, truth, _ = shapes_text(oracle, variant, m, 5)
    n = text.size
    td = to_dev(text, dev, misalign=5)
    cuts = [0, 7 * SEG - 5, 3 * ITEM + 11, BLOCK - 5 + 3, BLOCK + 32768 * 3 - 5, 3 * BLOCK + 999, 5 * BLOCK + 8100, n]
    wants, ends = [], []
    for k in range(len(cuts) - 1):
        lo, hi = cuts[k], cuts[k + 1]
        part = truth[(truth >= lo) & (truth < hi)]
        wants.append(part - lo + (k << 40) + lo)         # pos_base of piece k: its offset + k * 2^40
        ends.append(sum(w.size for w in wants))
    want = np.concatenate(wants)
    C = want.size
    caps = sorted({c + d for c in ends for d in (-1, 0, 1) if c + d >= 0} | {0, 1})
    sc = bmx.Scanner(0)
    st = torch.cuda.current_stream().cuda_stream
    sc.set_pattern(pat, variant, stream=st)
    want_d = torch.from_numpy(want).to(dev)
    for cap in caps:
        buf = guarded(G + cap + G, dev)
        ok(bmx, lib.bmx_scanner_begin(sc._h, c_void_p(buf.data_ptr() + 8 * G), cap, c_void_p(st)))
        for k in range(len(cuts) - 1):
            lo, hi = cuts[k], min(cuts[k + 1] + m - 1, n)
            ok(bmx, lib.bmx_scanner_scan(sc._h, c_void_p(td[lo:hi].data_ptr()), hi - lo, c_int64((k << 40) + lo), c_void_p(st)))
        count, _ = sc.finish(st)
        assert count == C, (label, cap, count, C)
        k = min(C, cap)
        exp = guarded(buf.numel(), dev)
        exp[G:G + k] = want_d[:k]
        if not torch.equal(buf, exp):
            assert_same(buf.cpu().numpy(), exp.cpu().numpy(), (label, "chain cap", cap))
        if cap in (ends[2] - 1, C + 1):                  # the result held by a cut list and by a complete one
            held = min(C, cap)
            for head in sorted({0, 1, max(held - 1, 0), held, held + 3}):
                dst = guarded(G + 2 + head + G, dev)
                ok(bmx, lib.bmx_scanner_export_result(sc._h, c_void_p(dst.data_ptr() + 8 * G), head, c_void_p(st)))
                got = dst.cpu().numpy()
                j = min(head, held)
                assert got[G] == C and got[G + 1] == held, (label, cap, head, got[G:G + 2])
                assert_same(got[G + 2:G + 2 + j], want[:j], (label, "export prefix", cap, head))
                assert_same(np.concatenate([got[:G], got[G + 2 + head:]]), np.full(2 * G, SENT), (label, "export guard", cap, head))
    sc.close()


def host_guarded(cap: int, off: int = G):
    return np.full(off + cap + G, SENT, dtype=np.int64)


def search_ex_guarded(bmx, text: np.ndarray, pat: bytes, variant: str, cap: int, off: int = G):
    buf = host_guarded(cap, off)
    count = c_uint64()
    ok(bmx, lib_of(bmx).bmx_search_ex(0, c_void_p(text.ctypes.data), text.size, pat, len(pat),
                                      c_void_p(buf.ctypes.data + 8 * off), cap, byref(count), VARIANT_IDS[variant], None))
    return count.value, buf


@pytest.mark.gpu
@pytest.mark.parametrize("label,variant,m", [VARIANTS[0], VARIANTS[3]], ids=["window-m1", "qgram-m7"])
def test_host_ingest_caps_at_chunk_seams(bmx, oracle, dev, monkeypatch, label, variant, m):  # noqa: F811
    """bmx_search_ex in 256 KiB chunks, resident and through the ring: caps at every chunk's cumulative count +-1;
    then the one-stream small-text path around its 8192-entry speculative read-back."""
    pat = b"a" * m
    text, truth, _ = shapes_text(oracle, variant, m, 0)
    chunk = 256 << 10
    C = truth.size
    ends = [int(np.searchsorted(truth, k * chunk - m + 1)) for k in range(1, -(-text.size // chunk))] + [C]
    caps = sorted({c + d for c in ends for d in (-1, 0, 1) if c + d >= 0} | {0, 1})
    monkeypatch.setenv("BMX_H2D_CHUNK_KB", "256")
    for resident in ("1000", "0"):
        monkeypatch.setenv("BMX_RESIDENT_MAX_MB", resident)
        for cap in caps:
            count, buf = search_ex_guarded(bmx, text, pat, variant, cap)
            assert count == C, (label, resident, cap, count)
            assert_same(buf, expect(buf.size, [(G, truth[:cap])]), (label, "ingest", resident, cap))
    monkeypatch.delenv("BMX_H2D_CHUNK_KB")
    monkeypatch.delenv("BMX_RESIDENT_MAX_MB")
    small = text[: 4 << 20]                             # kSmallHostBytes: one stream, the first 8192 positions ride along
    want = truth[truth <= small.size - m]
    assert want.size > 8193
    for cap in (0, 1, 8191, 8192, 8193, want.size - 1, want.size, want.size + 1):
        count, buf = search_ex_guarded(bmx, small, pat, variant, cap, G + 1)
        assert count == want.size, (label, "small", cap, count)
        assert_same(buf, expect(buf.size, [(G + 1, want[:cap])]), (label, "small", cap))


# ---------------------------------------------------------------------------------------------------------------
# Multi-pattern: a cap per pattern, outputs back to back between guard bands
# ---------------------------------------------------------------------------------------------------------------
def multi_text(oracle):
    """3 MB over 'bcd' with a 200 000-byte run of 'a' at the front (every start in it matches 'a' * 7) and three
    patterns planted behind it; the last one only late in the text."""
    rng = np.random.default_rng(77)
    n = 3_000_003
    text = rng.integers(98, 101, size=n, dtype=np.uint8)
    text[100:200_100] = ord("a")
    p1, p2, p3 = b"bcdbcdbbc", b"dcbdcbddcbcb", b"cbdcbdccbdbdcbdcbdcbbbcdcbdcbd"
    for i in range(40):
        for p, at in ((p1, 300_000 + 61_111 * i), (p2, 250_000 + 65_537 * i + 9)):
            text[at:at + len(p)] = np.frombuffer(p, dtype=np.uint8)
    for at in (2_500_001, 2_600_000, n - len(p3)):
        text[at:at + len(p3)] = np.frombuffer(p3, dtype=np.uint8)
    return text, [b"a" * 7, p1, p2, p3]


def run_multi(bmx, text, td, pats, caps, host: bool):
    """bmx_search_multi(_device) with caps[k] None (NULL output) or an int (0 included, with a non-NULL pointer).
    All outputs live in one allocation, G sentinel entries between neighbours, so an overflow of pattern k lands in
    the guard in front of pattern k + 1.  Returns (counts, buffer, offsets)."""
    lib = lib_of(bmx)
    K = len(pats)
    offs, size = [], G
    for cap in caps:
        offs.append(None if cap is None else size)
        size += 0 if cap is None else cap + G
    size += 4096                                        # slack: a list written with another pattern's cap stays inside
    buf = np.full(size, SENT, dtype=np.int64) if host else guarded(size, td.device)
    base = buf.ctypes.data if host else buf.data_ptr()
    c_pats = (ctypes.c_char_p * K)(*pats)
    c_ms = (ctypes.c_int32 * K)(*[len(p) for p in pats])
    c_pos = (c_void_p * K)(*[None if o is None else base + 8 * o for o in offs])
    c_caps = (c_int64 * K)(*[0 if c is None else c for c in caps])
    counts = (c_uint64 * K)()
    if host:
        ok(bmx, lib.bmx_search_multi(0, c_void_p(text.ctypes.data), text.size, K, c_pats, c_ms, c_pos, c_caps, counts))
    else:
        ok(bmx, lib.bmx_search_multi_device(c_void_p(td.data_ptr()), td.numel(), K, c_pats, c_ms, c_pos, c_caps, counts,
                                            stream_ptr()))
        buf = buf.cpu().numpy()
    return [int(c) for c in counts], buf, offs


@pytest.mark.gpu
def test_multi_pattern_caps_per_pattern(bmx, oracle, dev):  # noqa: F811
    """Different caps per pattern (NULL, 0 with a pointer, 1, c-1, c, c+1, a cap far above another pattern's count),
    on an eligible set, on an ineligible one (a three-byte pattern) and on the set that makes the union list too short
    for a late sparse pattern (a dense early pattern that only counts), device and host text."""
    text, pats = multi_text(oracle)
    td = to_dev(text, dev, misalign=3)
    ineligible = pats + [b"cdb"]
    for tag, ps in (("eligible", pats), ("ineligible", ineligible)):
        wants = [kmp(oracle, text, p) for p in ps]
        c = [w.size for w in wants]
        assert min(c) >= 3 and c[0] > 100_000
        vecs = [[None, c[1] - 1, 0, c[3] + 1], [c[0] + 1, 1, c[2], None], [0, c[1], c[2] - 1, 3],
                [c[0] - 1, c[1] + 1, 1, c[3]]]
        if tag == "eligible":
            # the union list of the first pass holds 3 entries, all from the run of 'a': pattern 3 gets none of its 3
            assert np.sort(np.concatenate(wants))[2] < wants[3][0]
            vecs.append([None, None, None, 3])
        else:
            vecs = [v + [x] for v, x in zip(vecs, (c[4] - 1, None, 2, 0))]
        for host in (False, True):
            for caps in vecs:
                counts, buf, offs = run_multi(bmx, text, td, ps, caps, host)
                assert counts == c, (tag, host, caps, counts, c)
                spans = [(o, w[:cap]) for o, w, cap in zip(offs, wants, caps) if o is not None]
                assert_same(buf, expect(buf.size, spans), (tag, "host" if host else "device", caps))


# ---------------------------------------------------------------------------------------------------------------
# Exchange collect and the multi-GPU searches
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("head_cap,tail_cap", [(8, 64), (4, 8)], ids=["whole-list", "prefix"])
def test_exchange_collect_out_cap_guards(bmx, oracle, dev, head_cap, tail_cap):  # noqa: F811
    """Three ranks on device 0 (one stream each), one step per out_cap: caps at every rank's cumulative count +-1,
    at the gathered prefix +-1, 1 and 0 with a pointer.  The gathered list is min(prefix, out_cap) long and nothing
    else in the guarded buffer changes.  With 4 + 8 entries of transport per rank the prefix ends inside rank 0."""
    from parallel_implementation_of_string_matching_algorithms_opencl_b200 import distributed as bd
    from test_exchange_gpu import _expected_prefix, _make_text

    lib = lib_of(bmx)
    world, local_cap = 3, 1 << 12
    text, pat = _make_text(bmx, 400_003, 9, 8, "dna", 60, world)
    m = len(pat)
    want, counts, prefix = _expected_prefix(oracle, text, pat, world, head_cap, tail_cap, local_cap, 1 << 30)
    assert np.array_equal(want, kmp(oracle, text, pat))
    assert (prefix.size == want.size) == (head_cap + tail_cap >= max(counts)), (counts, prefix.size)
    ends = np.cumsum(counts)
    out_caps = sorted({int(c) + d for c in list(ends) + [prefix.size] for d in (-1, 0, 1) if c + d >= 0} | {0, 1})
    streams = [torch.cuda.Stream(device=dev) for _ in range(world)]
    shards, scanners, xs, pos = [], [], [], []
    for r in range(world):
        lo, hi = bd.shard_bounds(text.size, world, r)
        lo, end = bd.shard_read_range(text.size, m, lo, hi)
        shards.append((torch.from_numpy(text[lo:end].copy()).to(dev), lo))
        sc = bmx.Scanner(0)
        sc.set_pattern(pat, stream=streams[r].cuda_stream)
        scanners.append(sc)
        pos.append(torch.empty(local_cap, dtype=torch.int64, device=dev))
        xs.append(bmx.Exchange(0, r, world, dst=0, head_cap=head_cap, tail_cap=tail_cap, depth=3))
    bmx.Exchange.connect_local(xs)
    for out_cap in out_caps:
        out = guarded(G + out_cap + G, dev)
        torch.cuda.synchronize()
        for r in range(world):
            st = streams[r].cuda_stream
            scanners[r].begin(pos[r], stream=st)
            scanners[r].scan(shards[r][0], shards[r][1], stream=st)
            seq = xs[r].post(scanners[r], st)
        for r in range(world):
            ptr = c_void_p(out.data_ptr() + 8 * G) if r == 0 else None
            ok(bmx, lib.bmx_exchange_collect(xs[r]._h, ptr, out_cap if r == 0 else 0, c_void_p(streams[r].cuda_stream),
                                             byref(c_uint64())))
        got = [xs[r].wait(seq) for r in range(world)]
        torch.cuda.synchronize()
        k = min(prefix.size, out_cap)
        assert got[0][0] == want.size and got[0][1] == counts and got[0][2] == k, (out_cap, got[0])
        buf = out.cpu().numpy()
        assert_same(buf, expect(buf.size, [(G, prefix[:k])]), ("exchange", head_cap, tail_cap, out_cap))
    for x in xs:
        x.close()
    for sc in scanners:
        sc.close()


@pytest.mark.gpu
def test_multi_gpu_search_guards(bmx, oracle, dev):  # noqa: F811
    """bmx_mg_search_device (output on GPU 0) and bmx_mg_search (host output) on every visible GPU: caps at every
    shard's cumulative count +-1, 1, 0 with a pointer and the count +-1."""
    from parallel_implementation_of_string_matching_algorithms_opencl_b200 import distributed as bd
    from test_exchange_gpu import _make_text

    lib = lib_of(bmx)
    mg = bmx.MultiGpu(0)
    R = mg.ngpus
    text, pat = _make_text(bmx, 1_000_003, 12, 21, "dna", 80, R)
    text[100_000:160_000] = ord("C")
    pat = b"CCCCCCC"
    m = len(pat)
    want = kmp(oracle, text, pat)
    C = want.size
    shards, bases, ends = [], [], []
    for r in range(R):
        lo, hi = bd.shard_bounds(text.size, R, r)
        ends.append(int(np.searchsorted(want, hi)))
        lo, end = bd.shard_read_range(text.size, m, lo, hi)
        shards.append(torch.from_numpy(text[lo:end].copy()).to(torch.device("cuda", r)))
        bases.append(lo)
    caps = sorted({c + d for c in ends + [C] for d in (-1, 0, 1) if c + d >= 0} | {0, 1})
    ptrs = (c_void_p * R)(*[t.data_ptr() for t in shards])
    ns = (c_int64 * R)(*[t.numel() for t in shards])
    bs = (c_int64 * R)(*bases)
    for cap in caps:
        count, per = c_uint64(), (c_uint64 * R)()
        out = guarded(G + 1 + cap + G, dev)
        ok(bmx, lib.bmx_mg_search_device(mg._h, ptrs, ns, bs, pat, m, c_void_p(out.data_ptr() + 8 * (G + 1)), cap,
                                         byref(count), per))
        torch.cuda.synchronize()
        assert count.value == C and sum(per) == C, ("mg device", cap, count.value)
        buf = out.cpu().numpy()
        assert_same(buf, expect(buf.size, [(G + 1, want[:cap])]), ("mg device", cap))
        host = host_guarded(cap)
        ok(bmx, lib.bmx_mg_search(mg._h, c_void_p(text.ctypes.data), text.size, pat, m, c_void_p(host.ctypes.data + 8 * G),
                                  cap, byref(count), per))
        assert count.value == C, ("mg host", cap, count.value)
        assert_same(host, expect(host.size, [(G, want[:cap])]), ("mg host", cap))
    mg.close()
