"""Case-insensitive search (BMX_IGNORE_CASE): the result must be exactly the exact search's result for
text.lower() and pattern.lower() -- count, ascending positions, pos_cap truncation and pos_base -- on every filter
kind, emission path and host ingest layout, without writing the caller's text.  The truth is the oracle on the
lowered bytes (bytes.find on them for patterns beyond 2000 bytes, where the oracle's tables get slow)."""
from __future__ import annotations

import ctypes
import re
import zlib
from pathlib import Path

import numpy as np
import pytest

from test_parity_gpu import _find_all, dev, to_dev  # noqa: F401  (dev is a fixture)

torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]

LETTER_BOUNDARIES = b"@[`{"                      # the bytes on either side of 'A'..'Z' and 'a'..'z'
HIGH_TWINS = bytes(range(0xC1, 0xDB)) + bytes(range(0xE1, 0xFB))   # letters with bit 7 set: never folded


def set_knobs(monkeypatch, **knobs):
    for k, v in knobs.items():
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, str(v))


def truth(oracle, text, pat: bytes) -> np.ndarray:
    low, plow = bytes(text).lower(), pat.lower()
    if len(pat) <= 2000:
        return oracle.search(low, plow)
    return _find_all(low, plow)


def mixcase(pat: bytes, rng) -> bytes:
    """pat with every ASCII letter in a random case."""
    flip = rng.integers(0, 2, size=len(pat)).astype(bool)
    return bytes(c ^ 0x20 if f and chr(c).isascii() and chr(c).isalpha() else c for c, f in zip(pat, flip))


def check_ic(bmx, td, pat: bytes, want: np.ndarray, variant="auto", tag=()):
    """Full list, caps below the count, count-only; every call must report the case-folding kernels."""
    count, pos, stats = bmx.search_device(td, pat, max_positions=max(want.size, 1), variant=variant, ignore_case=True)
    assert count == want.size and np.array_equal(pos.cpu().numpy(), want), (*tag, "full", count, want.size)
    assert stats["ignore_case"], (*tag, stats)
    for cap in sorted({max(want.size // 2, 1), 1}):
        count, pos, _ = bmx.search_device(td, pat, max_positions=cap, variant=variant, ignore_case=True)
        assert count == want.size and np.array_equal(pos.cpu().numpy(), want[:cap]), (*tag, "cap", cap)
    count, pos, _ = bmx.search_device(td, pat, variant=variant, ignore_case=True)
    assert count == want.size and pos is None, (*tag, "count-only", count, want.size)
    return stats


def plant_seams(text: np.ndarray, pat: bytes, rng, tile: int = 16384, every: int = 5):
    """Mixed-case copies of pat at the text's ends and straddling tile seams (front, middle and last byte on the seam)."""
    n, m = text.size, len(pat)
    spots = [0, n - m]
    for s in range(tile, n - m, tile * every):
        spots += [s - m + 1, s - m // 2, s]
    for s in spots:
        if 0 <= s <= n - m:
            text[s:s + m] = np.frombuffer(mixcase(pat, rng), dtype=np.uint8)
    return text


# ---------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------
def test_ignore_case_constant_matches_header(bmx):
    header = (ROOT / "include" / "bmx.h").read_text()
    value = re.search(r"#define\s+BMX_IGNORE_CASE\s+(0x[0-9a-fA-F]+|\d+)", header)
    assert value, "BMX_IGNORE_CASE not defined in include/bmx.h"
    assert bmx._lib.IGNORE_CASE == int(value.group(1), 0)


# ---------------------------------------------------------------------------------------------------------------
# 1. Byte classes: '@' '[' '`' '{' and the letters with bit 7 set never match a letter
# ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("pat", [b"a", b"Z", b"aZ", b"zA1", b"AzaZ", b"aZ@zA", b"Zebra-AZaz", b"AZaz" * 4, b"zZaA[`" * 7])
def test_byte_class_boundaries(bmx, oracle, dev, pat):  # noqa: F811
    rng = np.random.default_rng(zlib.crc32(pat))
    n = (1 << 20) + 13
    text = rng.integers(0, 256, size=n, dtype=np.uint8)
    text[: 256 * 16] = np.tile(np.arange(256, dtype=np.uint8), 16)   # every byte value, many times
    m = len(pat)
    letters = [i for i, c in enumerate(pat) if chr(c).isalpha()]
    spot = 4096
    while spot + m < n - 64:
        text[spot:spot + m] = np.frombuffer(mixcase(pat, rng), dtype=np.uint8)
        # near misses: one letter replaced by a neighbour of the letter ranges or by its bit-7 twin
        bad = bytearray(mixcase(pat, rng))
        i = letters[int(rng.integers(0, len(letters)))]
        bad[i] = int(rng.choice(np.frombuffer(LETTER_BOUNDARIES + HIGH_TWINS + bytes([bad[i] | 0x80]), dtype=np.uint8)))
        text[spot + m + 7: spot + 2 * m + 7] = np.frombuffer(bytes(bad), dtype=np.uint8)
        spot += 9973
    want = truth(oracle, text.tobytes(), pat)
    assert want.size >= 50
    td = to_dev(text, dev, misalign=3)
    for variant in ["auto", "window", "qgram"] + (["shiftand"] if m <= 32 else []):
        check_ic(bmx, td, pat, want, variant, tag=(pat, variant))


# ---------------------------------------------------------------------------------------------------------------
# 2. Every filter kind and pattern length, with positions, count-only and caps below the count
# ---------------------------------------------------------------------------------------------------------------
LENGTHS = [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 16, 32, 33, 64, 1024, 1025, 4096, 4097, 5000]


@gpu
@pytest.mark.parametrize("m", LENGTHS)
def test_every_kind_and_length(bmx, oracle, dev, m):  # noqa: F811
    rng = np.random.default_rng(1000 + m)
    alpha = np.frombuffer(b"abcdeABCDE-. xyzXYZ", dtype=np.uint8)   # mixed case, so the filters see candidates
    n = (2 << 20) + 7 if m <= 64 else (1 << 20) + 7
    text = alpha[rng.integers(0, alpha.size, size=n)].astype(np.uint8)
    pat = mixcase(bytes(alpha[rng.integers(0, alpha.size, size=m)]), rng)
    if not any(chr(c).isalpha() for c in pat):
        pat = b"q" + pat[1:]
    plant_seams(text, pat, rng, tile=16384, every=3)
    want = truth(oracle, text.tobytes(), pat)
    assert want.size >= 2
    td = to_dev(text, dev)
    for variant in ["auto", "qgram", "window"] + (["shiftand"] if m <= 32 else []):
        check_ic(bmx, td, pat, want, variant, tag=(m, variant))


# kBytes5 (m = 5, 6 on few distinct bytes) and kQgramPerResidue (7 <= m <= 9 on small alphabets), both ways, and the
# per-lane verification that BMX_COOP_VERIFY=0 selects, on mixed-case DNA
DNA_KNOBS = [
    (5, "window", {"BMX_WINDOW5": 1}), (6, "window", {"BMX_WINDOW5": 1}),
    (5, "window", {"BMX_WINDOW5": 0}), (6, "window", {"BMX_WINDOW5": 0}),
    (7, "qgram", {"BMX_QGRAM_UNIFORM": 0}), (8, "qgram", {"BMX_QGRAM_UNIFORM": 0}), (9, "qgram", {"BMX_QGRAM_UNIFORM": 0}),
    (7, "qgram", {"BMX_QGRAM_UNIFORM": 1}), (9, "qgram", {"BMX_QGRAM_UNIFORM": 1}),
    (12, "qgram", {"BMX_COOP_VERIFY": 0}), (40, "window", {"BMX_COOP_VERIFY": 0}), (7, "qgram", {"BMX_COOP_VERIFY": 0, "BMX_QGRAM_UNIFORM": 0}),
]


@gpu
@pytest.mark.parametrize("m,variant,knobs", DNA_KNOBS, ids=[f"m{m}-{v}-" + "-".join(f"{k}{x}" for k, x in kn.items()) for m, v, kn in DNA_KNOBS])
def test_mixed_case_dna_knobs(bmx, oracle, dev, monkeypatch, m, variant, knobs):  # noqa: F811
    set_knobs(monkeypatch, **knobs)
    rng = np.random.default_rng(m * 31 + len(knobs))
    alpha = np.frombuffer(b"ACGTacgt", dtype=np.uint8)
    text = alpha[rng.integers(0, 8, size=(1 << 20) + 5)].astype(np.uint8)
    pat = mixcase(bytes(alpha[rng.integers(0, 4, size=m)]), rng)
    plant_seams(text, pat, rng)
    want = truth(oracle, text.tobytes(), pat)
    td = to_dev(text, dev, misalign=7)
    check_ic(bmx, td, pat, want, variant, tag=(m, variant, knobs))


# ---------------------------------------------------------------------------------------------------------------
# 3. Dense text: every start position matches (dense tile path, full segments in the expand kernel)
# ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("pat", [b"AA", b"aAa", b"AaAAaaAaaAAaAaaaAAaaAaAa"])
def test_dense_text(bmx, dev, pat):  # noqa: F811
    n = (3 << 20) + 6
    text = np.resize(np.frombuffer(b"aA", dtype=np.uint8), n)
    want = np.arange(n - len(pat) + 1, dtype=np.int64)
    td = to_dev(text, dev)
    for variant in ["auto", "window"] + (["qgram"] if len(pat) >= 7 else []):
        count, pos, stats = bmx.search_device(td, pat, max_positions=n, variant=variant, ignore_case=True)
        assert count == want.size and np.array_equal(pos.cpu().numpy(), want), (pat, variant)
        count, _, _ = bmx.search_device(td, pat, variant=variant, ignore_case=True)
        assert count == want.size
        count, pos, _ = bmx.search_device(td, pat, max_positions=5000, variant=variant, ignore_case=True)
        assert count == want.size and np.array_equal(pos.cpu().numpy(), want[:5000])
    # the exact search: the text has period 2, so the pattern matches at every even or every odd start, or nowhere
    m = len(pat)
    starts = np.arange(n - m + 1)
    want_exact = sum(int(np.count_nonzero(starts % 2 == r)) for r in (0, 1) if text[r:r + m].tobytes() == pat)
    assert bmx.search_device(td, pat)[0] == want_exact


# ---------------------------------------------------------------------------------------------------------------
# 4. Boundaries: tile seams at both tile sizes, device offsets 1..15, ragged ends, first and last start, m = 70 000
# ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("tile", [16384, None])
def test_tile_seams_offsets_and_ragged_ends(bmx, oracle, dev, monkeypatch, tile):  # noqa: F811
    set_knobs(monkeypatch, BMX_TILE=tile)
    rng = np.random.default_rng(77 if tile else 78)
    alpha = np.frombuffer(bytes(range(0x20, 0x7F)), dtype=np.uint8)
    for m in (3, 7, 16, 33):
        pat = mixcase(bytes(alpha[rng.integers(0, alpha.size, size=m)]), rng)
        if not any(chr(c).isalpha() for c in pat):
            pat = b"K" + pat[1:]
        n = (1 << 20) + 16 * m + 9                     # not a multiple of 16: the producer copies a ragged tail
        text = alpha[rng.integers(0, alpha.size, size=n)].astype(np.uint8)
        plant_seams(text, pat, rng, tile=tile or 32768, every=2)
        want = truth(oracle, text.tobytes(), pat)
        assert want[0] == 0 and want[-1] == n - m
        for misalign in range(0, 16):
            td = to_dev(text, dev, misalign=misalign)
            count, pos, _ = bmx.search_device(td, pat, max_positions=want.size, pos_base=1000, ignore_case=True)
            assert count == want.size and np.array_equal(pos.cpu().numpy(), want + 1000), (m, misalign)
        check_ic(bmx, to_dev(text, dev, misalign=9), pat, want, tag=(m, "misalign 9"))


@gpu
def test_pattern_verified_from_global_memory(bmx, dev):  # noqa: F811
    """m = 70 000 > 4096: candidates are verified from the caller's text in global memory, which is never folded."""
    rng = np.random.default_rng(70000)
    alpha = np.frombuffer(b"abcdefgABCDEFG0123", dtype=np.uint8)
    m, n = 70000, (1 << 20) + 3
    text = alpha[rng.integers(0, alpha.size, size=n)].astype(np.uint8)
    pat = bytes(alpha[rng.integers(0, alpha.size, size=m)])
    for s in (0, 300001, 400003, 655360 - 7, n - m):
        text[s:s + m] = np.frombuffer(mixcase(pat, rng), dtype=np.uint8)
    near = bytearray(mixcase(pat, rng))
    near[m // 2] = ord("@") if chr(near[m // 2]).isalpha() else ord("Q")
    text[500000:500000 + m] = np.frombuffer(bytes(near), dtype=np.uint8)
    want = _find_all(text.tobytes().lower(), pat.lower())
    assert want.size == 5
    for variant in ("auto", "window", "qgram"):
        check_ic(bmx, to_dev(text, dev, misalign=5), mixcase(pat, rng), want, variant, tag=(variant,))


# ---------------------------------------------------------------------------------------------------------------
# 5. The pattern cache keys on the flag, on every host path
# ---------------------------------------------------------------------------------------------------------------
def abc_text(n: int) -> bytes:
    """Filler without 'abc' in any case, with one 'abc', one 'ABC' and one 'Abc', the last two across 64 KiB seams."""
    rng = np.random.default_rng(3)
    filler = np.frombuffer(b"xyzXYZ-_ 0123", dtype=np.uint8)
    t = filler[rng.integers(0, filler.size, size=n)].astype(np.uint8)
    for off, w in ((1000, b"abc"), ((64 << 10) - 1, b"ABC"), ((192 << 10) - 2, b"Abc")):
        t[off:off + 3] = np.frombuffer(w, dtype=np.uint8)
    return t.tobytes()


ABC_ROUNDS = [(b"Abc", False, [(192 << 10) - 2]), (b"Abc", True, [1000, (64 << 10) - 1, (192 << 10) - 2]),
              (b"Abc", False, [(192 << 10) - 2]), (b"aBC", True, [1000, (64 << 10) - 1, (192 << 10) - 2])]


@gpu
@pytest.mark.parametrize("layout", ["small", "chunked", "ring"])
def test_cache_keys_on_flag_host_paths(bmx, dev, monkeypatch, layout):  # noqa: F811
    knobs = {"small": {}, "chunked": {"BMX_SMALL_HOST": 0, "BMX_H2D_CHUNK_KB": 64},
             "ring": {"BMX_RESIDENT_MAX_MB": 0, "BMX_H2D_CHUNK_KB": 64}}[layout]
    set_knobs(monkeypatch, **knobs)
    text = abc_text(1 << 20)
    for _ in range(2):
        for pat, ic, want in ABC_ROUNDS:
            count, pos, stats = bmx.search(text, pat, ignore_case=ic, return_stats=True)
            assert count == len(want) and pos.tolist() == want, (layout, pat, ic, count)
            assert stats["ignore_case"] == ic
            count, _ = bmx.search(text, pat, max_positions=0, ignore_case=ic)
            assert count == len(want)


@gpu
def test_cache_keys_on_flag_device_two_streams(bmx, dev):  # noqa: F811
    td = to_dev(abc_text(1 << 20), dev, misalign=1)
    streams = [torch.cuda.Stream(dev), torch.cuda.Stream(dev)]
    torch.cuda.synchronize(dev)
    for k in range(3):
        for i, (pat, ic, want) in enumerate(ABC_ROUNDS):
            s = streams[(i + k) % 2]
            count, pos, stats = bmx.search_device(td, pat, max_positions=8, ignore_case=ic, stream=s)
            torch.cuda.synchronize(dev)
            assert count == len(want) and pos.cpu().tolist() == want, (k, pat, ic)
            assert stats["ignore_case"] == ic


# ---------------------------------------------------------------------------------------------------------------
# 6. Flag reporting and argument checks
# ---------------------------------------------------------------------------------------------------------------
@gpu
def test_flag_reporting_and_bad_variants(bmx, oracle, dev):  # noqa: F811
    rng = np.random.default_rng(6)
    alpha = np.frombuffer(b"0123-+@[`{ aAzZ", dtype=np.uint8)
    text = alpha[rng.integers(0, alpha.size, size=(1 << 20) + 1)].astype(np.uint8)
    td = to_dev(text, dev)
    for pat in (b"12", b"0-3+", b"@[`{", b"1230-+12"):   # no ASCII letter: the flag is dropped, exact kernels run
        want = oracle.search(text.tobytes(), pat)
        for variant in ("auto", "window", "qgram"):
            count, pos, stats = bmx.search_device(td, pat, max_positions=want.size + 1, variant=variant, ignore_case=True)
            assert count == want.size and np.array_equal(pos.cpu().numpy(), want)
            _, _, exact = bmx.search_device(td, pat, variant=variant)
            assert not stats["ignore_case"] and stats["variant"] == exact["variant"], (pat, variant, stats)
    for pat in (b"a", b"1z", b"Z@a`", b"0aZ12345"):
        _, _, stats = bmx.search_device(td, pat, ignore_case=True)
        _, _, exact = bmx.search_device(td, pat)
        assert stats["ignore_case"] and stats["variant"] == exact["variant"]
        raw = bmx._lib.BmxStats()
        cnt = ctypes.c_uint64()
        bmx._lib.check(bmx._lib.load().bmx_search_device_ex(ctypes.c_void_p(td.data_ptr()), td.numel(), pat, len(pat), 0, None, 0,
                                                            ctypes.byref(cnt), bmx._lib.VARIANT_AUTO | bmx._lib.IGNORE_CASE,
                                                            ctypes.byref(raw), None))
        assert raw.variant & ~bmx._lib.IGNORE_CASE == {"qgram": 1, "window": 2, "shiftand": 3}[exact["variant"]]
        assert raw.variant & bmx._lib.IGNORE_CASE
    host = text[:4096].tobytes()
    sc = bmx.Scanner(0)
    for variant in (0x200, 0x104, 0x100 | 7, 0x300, 0x1101, -1, 0x100 | -4):
        with pytest.raises(bmx._lib.BmxError) as e:
            bmx.search(host, b"aZ", variant=variant)
        assert e.value.code == bmx._lib.BMX_E_BADARG, variant
        with pytest.raises(bmx._lib.BmxError) as e:
            bmx.search_device(td, b"aZ", variant=variant)
        assert e.value.code == bmx._lib.BMX_E_BADARG, variant
        with pytest.raises(bmx._lib.BmxError) as e:
            sc.set_pattern(b"aZ", variant=variant)
        assert e.value.code == bmx._lib.BMX_E_BADARG, variant
    sc.close()
    # the library stays usable
    assert bmx.search(b"xAzx", b"az", ignore_case=True)[0] == 1


# ---------------------------------------------------------------------------------------------------------------
# 7. The caller's device text is left as it was
# ---------------------------------------------------------------------------------------------------------------
@gpu
def test_device_text_unchanged(bmx, dev):  # noqa: F811
    rng = np.random.default_rng(7)
    text = rng.integers(0, 256, size=(4 << 20) + 3, dtype=np.uint8)
    td = to_dev(text, dev, misalign=2)
    before = td.clone()
    for pat in (b"Q", b"aB", b"XyZw", b"Hello", b"HeLLo World", b"A" * 40, b"mIxEd" * 1000):
        for variant in ("auto", "window", "qgram", "shiftand"):
            bmx.search_device(td, pat, max_positions=16, variant=variant, ignore_case=True)
    torch.cuda.synchronize(dev)
    assert torch.equal(td, before)


# ---------------------------------------------------------------------------------------------------------------
# 8. Chained scans over consecutive chunks with (m - 1)-byte halos equal one search
# ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("m", [2, 9, 33])
def test_chained_scans(bmx, oracle, dev, m):  # noqa: F811
    rng = np.random.default_rng(800 + m)
    alpha = np.frombuffer(b"aAbBcC", dtype=np.uint8)
    n = (3 << 20) + 11
    text = alpha[rng.integers(0, alpha.size, size=n)].astype(np.uint8)
    pat = mixcase(b"abcabcabcabcabcabcabcabcabcabcabcabc"[:m], rng)
    plant_seams(text, pat, rng)
    want = truth(oracle, text.tobytes(), pat)
    td = to_dev(text, dev)
    cuts = [0, 12345, 12346 + m, 1 << 20, (1 << 20) + 32768 * 3 + 5, n]
    sc = bmx.Scanner(0)
    for cap in (want.size, max(want.size // 3, 1)):
        out = torch.full((cap + 8,), -7, dtype=torch.int64, device=dev)
        sc.set_pattern(pat, ignore_case=True)
        sc.begin(out[:cap])
        for a, b in zip(cuts[:-1], cuts[1:]):
            end = min(b + m - 1, n)
            sc.scan(td[a:end], pos_base=a)
        count, stats = sc.finish()
        assert stats["ignore_case"]
        assert count == want.size
        got = out.cpu().numpy()
        assert np.array_equal(got[:cap], want[:cap]) and np.all(got[cap:] == -7), (m, cap)
    sc.close()


# ---------------------------------------------------------------------------------------------------------------
# 9. Full size: 1 GiB of upper-case DNA, a lower-case pattern
# ---------------------------------------------------------------------------------------------------------------
@gpu
def test_full_size_dna(bmx, oracle, dev):  # noqa: F811
    n, m, seed = 1 << 30, 32, 9
    alpha = bmx.synth.ALPHABETS["dna"]
    td = torch.empty(n, dtype=torch.uint8, device=dev)
    bmx.synth.fill_device(td, 0, seed, alpha)
    pat = bmx.synth.pattern_from_stream(m, seed, alpha)
    bmx.synth.plant_device(td, pat, bmx.synth.plant_offsets(n, m, 5000, seed))
    torch.cuda.synchronize(dev)
    want = oracle.search_np(td.cpu().numpy(), pat)
    assert want.size >= 4000
    cap = want.size + 16
    c_ic, p_ic, s_ic = bmx.search_device(td, pat.lower(), max_positions=cap, ignore_case=True)
    c_ex, p_ex, s_ex = bmx.search_device(td, pat, max_positions=cap)
    assert s_ic["ignore_case"] and not s_ex["ignore_case"]
    assert c_ic == c_ex == want.size
    assert np.array_equal(p_ic.cpu().numpy(), want) and np.array_equal(p_ex.cpu().numpy(), want)
    assert bmx.search_device(td, pat.lower(), ignore_case=True)[0] == want.size
    assert bmx.search_device(td, pat.lower())[0] == 0
