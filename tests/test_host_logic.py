"""CPU: host-side logic of libbmx.so (tables, word partitioner) against the reference's own
tables (golden), the reference code when built here, and the oracle; plus the ABI surface:
the library loads, exports every symbol include/bmx.h declares, and rejects bad arguments.
No compute call needs a GPU here."""
from __future__ import annotations

import ctypes
import random
import re
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]


def test_library_exports_every_declared_symbol(bmx):
    header = (ROOT / "include" / "bmx.h").read_text()
    declared = set(re.findall(r"\b(bmx_[a-z_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    lib = bmx._lib.load()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/bmx.h but not exported"
    assert declared == set(bmx._lib.EXPORTS)
    assert bmx.version() == 200


def test_tables_equal_reference_tables(bmx, golden):
    for pat, bad128, good in golden.tables():
        bad, g = bmx.build_tables(pat)
        assert np.array_equal(bad[:128], bad128), pat
        assert np.all(bad[128:] == len(pat))          # widened half: bytes >= 0x80 not in the pattern
        assert np.array_equal(g[1:], good[1:]), pat     # good[0] is unused by the reference
        assert g[0] == 0


def test_tables_equal_oracle_fuzz(bmx, oracle):
    rnd = random.Random(11)
    for it in range(3000):
        sigma = rnd.choice([1, 2, 2, 3, 4, 26, 256])
        m = rnd.randint(1, 40) if it % 10 else rnd.randint(100, 700)
        if rnd.random() < 0.3:   # periodic patterns exercise the border cases
            unit = bytes(rnd.randrange(sigma) for _ in range(rnd.randint(1, 5)))
            pat = (unit * (m // len(unit) + 1))[:m]
        else:
            pat = bytes(rnd.randrange(sigma) for _ in range(m))
        bad, good = bmx.build_tables(pat)
        obad, ogood = oracle.tables(pat)
        assert np.array_equal(bad, obad), pat
        assert np.array_equal(good[1:], ogood[1:]), pat


def test_tables_equal_reference_code_fuzz(bmx, reflib):
    rnd = random.Random(5)
    for _ in range(5000):
        sigma = rnd.randint(1, 5)
        m = rnd.randint(1, 99)
        pat = bytes(rnd.randrange(97, 97 + sigma) for _ in range(m))
        bad128 = np.zeros(128, dtype=np.int32)
        rgood = np.zeros(m + 1, dtype=np.int32)
        assert reflib.ref_bm_build_tables(ctypes.c_char_p(pat), m, bad128.ctypes.data_as(ctypes.c_void_p),
                                          rgood.ctypes.data_as(ctypes.c_void_p)) == 0
        bad, good = bmx.build_tables(pat)
        assert np.array_equal(bad[:128], bad128) and np.array_equal(good[1:], rgood[1:m]), pat


def test_long_pattern_tables_are_linear_time(bmx, oracle):
    m = 1 << 20
    pat = (b"ab" * (m // 2))[:-1] + b"c"
    bad, good = bmx.build_tables(pat)           # the reference's O(m^3) walk would never finish
    assert bad[ord("a")] == 1 and bad[ord("b")] == 2 and bad[ord("c")] == m
    assert good[1] == m and good[m - 1] == m
    small = pat[-600:]
    assert np.array_equal(bmx.build_tables(small)[1][1:], oracle.tables(small)[1][1:])


def test_partitioner_matches_reference_and_oracle(bmx, oracle, golden):
    for name, _pat, nparts, se, _ans in golden.parts():
        assert np.array_equal(bmx.partition_words(golden.text(name), nparts), se), name
    rnd = random.Random(3)
    for _ in range(2000):
        n = rnd.randint(1, 120)
        text = bytes(rnd.choice(b"ab c") for _ in range(n))   # leading / doubled spaces included
        for nparts in (1, 2, 3, 5):
            assert np.array_equal(bmx.partition_words(text, nparts), oracle.partition_words(text, nparts)), (text, nparts)
    t = golden.text("input5L")
    for nparts in (1, 2, 3, 4, 7, 10):
        assert np.array_equal(bmx.partition_words(t, nparts), oracle.partition_words(t, nparts))


def test_bad_arguments_are_rejected_without_touching_a_gpu(bmx):
    lib = bmx._lib.load()
    E = bmx._lib
    bad = (ctypes.c_int32 * 256)()
    good = (ctypes.c_int32 * 8)()
    assert lib.bmx_build_tables(b"abc", 0, bad, good) == E.BMX_E_BADARG          # empty pattern
    assert lib.bmx_build_tables(None, 3, bad, good) == E.BMX_E_BADARG
    assert b"m" in lib.bmx_last_error()
    cnt = ctypes.c_uint64()
    # m <= 0 is rejected before any device work (the reference would report n+1 bogus hits)
    assert lib.bmx_search_ex(0, b"abc", 3, b"", 0, None, 0, ctypes.byref(cnt), 0, None) in (E.BMX_E_BADARG, E.BMX_E_NODEVICE)
    assert lib.bmx_search_ex(0, b"abc", -1, b"a", 1, None, 0, ctypes.byref(cnt), 0, None) == E.BMX_E_BADARG
    assert lib.bmx_search_ex(0, b"abc", 3, b"a", 1, None, 0, None, 0, None) == E.BMX_E_BADARG
    se = (ctypes.c_int32 * 2)(0, 2)
    ans = (ctypes.c_int32 * 1)()
    assert lib.bmx_search_partitions(b"abc", b"", se, ans, None, None, 0, 1) == E.BMX_E_BADARG
    wrong_gs = (ctypes.c_int32 * 2)(0, 7)
    assert lib.bmx_search_partitions(b"abcab", b"ab", se, ans, wrong_gs, None, 2, 1) == E.BMX_E_TABLES
    assert lib.bmx_partition_words(b"a b", 3, 0, se) == E.BMX_E_BADARG

    # The other entry points, one bad argument each.  BADARG alone where the check comes before the device lookup;
    # BADARG or NODEVICE where it comes after (a machine without a GPU stops at the lookup).
    either = (E.BMX_E_BADARG, E.BMX_E_NODEVICE)
    first = ctypes.c_int64()
    assert lib.bmx_search_device_ex(None, -1, b"a", 1, 0, None, 0, ctypes.byref(cnt), 0, None, None) == E.BMX_E_BADARG
    assert lib.bmx_search_device_ex(None, 0, b"a", 1, 0, None, 0, None, 0, None, None) == E.BMX_E_BADARG
    assert lib.bmx_search_device_ex(None, 0, b"a", 1, 0, None, -1, ctypes.byref(cnt), 0, None, None) == E.BMX_E_BADARG
    assert lib.bmx_search_device_ex(None, 0, b"", 0, 0, None, 0, ctypes.byref(cnt), 0, None, None) in either
    assert lib.bmx_find_first_device(None, -1, b"a", 1, ctypes.byref(first), None) == E.BMX_E_BADARG
    assert lib.bmx_find_first_device(None, 0, b"a", 1, None, None) == E.BMX_E_BADARG
    assert lib.bmx_find_first_device(None, 0, b"", 0, ctypes.byref(first), None) in either
    assert lib.bmx_find_first(b"abc", -1, b"a", 1, ctypes.byref(first)) == E.BMX_E_BADARG
    assert lib.bmx_find_first(b"abc", 3, b"a", 1, None) == E.BMX_E_BADARG
    assert lib.bmx_find_first(b"abc", 3, b"", 0, ctypes.byref(first)) == E.BMX_E_BADARG

    pats = (ctypes.c_char_p * 2)(b"ab", None)   # a NULL pattern in the set
    ms = (ctypes.c_int32 * 2)(2, 2)
    ms0 = (ctypes.c_int32 * 2)(2, 0)
    good_pats = (ctypes.c_char_p * 2)(b"ab", b"cd")
    counts = (ctypes.c_uint64 * 2)()
    multi_host = lambda *a: lib.bmx_search_multi(0, *a)              # noqa: E731
    multi_device = lambda *a: lib.bmx_search_multi_device(*a, None)  # noqa: E731
    for fn in (multi_host, multi_device):
        assert fn(b"abcd", 4, 2, pats, ms, None, None, counts) == E.BMX_E_BADARG
        assert fn(b"abcd", 4, 2, good_pats, ms0, None, None, counts) == E.BMX_E_BADARG
        assert fn(b"abcd", -1, 2, good_pats, ms, None, None, counts) == E.BMX_E_BADARG
        assert fn(b"abcd", 4, -1, good_pats, ms, None, None, counts) == E.BMX_E_BADARG
        assert fn(b"abcd", 4, 2, good_pats, ms, None, None, None) == E.BMX_E_BADARG

    # a zeroed block stands in for a bmx_mg handle: these calls reject their arguments before they read it
    mg = ctypes.create_string_buffer(256)
    shard_counts = (ctypes.c_uint64 * 1)()
    assert lib.bmx_mg_search(None, b"abc", 3, b"a", 1, None, 0, ctypes.byref(cnt), shard_counts) == E.BMX_E_BADARG
    assert lib.bmx_mg_search(mg, b"abc", -1, b"a", 1, None, 0, ctypes.byref(cnt), shard_counts) == E.BMX_E_BADARG
    assert lib.bmx_mg_search(mg, b"abc", 3, b"", 0, None, 0, ctypes.byref(cnt), shard_counts) == E.BMX_E_BADARG
    assert lib.bmx_mg_search(mg, b"abc", 3, b"a", 1, None, -1, ctypes.byref(cnt), shard_counts) == E.BMX_E_BADARG
    texts = (ctypes.c_void_p * 1)()
    lens = (ctypes.c_int64 * 1)(3)
    bases = (ctypes.c_int64 * 1)(0)
    assert lib.bmx_mg_search_device(None, texts, lens, bases, b"a", 1, None, 0, ctypes.byref(cnt), shard_counts) == E.BMX_E_BADARG
    assert lib.bmx_mg_search_device(mg, None, lens, bases, b"a", 1, None, 0, ctypes.byref(cnt), shard_counts) == E.BMX_E_BADARG
    assert lib.bmx_mg_search_device(mg, texts, lens, bases, b"", 0, None, 0, ctypes.byref(cnt), shard_counts) == E.BMX_E_BADARG
    assert lib.bmx_mg_search_device(mg, texts, lens, bases, b"a", 1, None, -1, ctypes.byref(cnt), shard_counts) == E.BMX_E_BADARG

    handle = ctypes.c_void_p()
    assert lib.bmx_exchange_create(0, 0, 1, 0, 0, 0, 2, None) == E.BMX_E_BADARG
    assert lib.bmx_exchange_create(0, 0, 0, 0, 0, 0, 2, ctypes.byref(handle)) == E.BMX_E_BADARG   # world 0
    assert lib.bmx_exchange_create(0, 1, 1, 0, 0, 0, 2, ctypes.byref(handle)) == E.BMX_E_BADARG   # rank >= world
    assert lib.bmx_exchange_create(0, 0, 1, 0, -1, 0, 2, ctypes.byref(handle)) == E.BMX_E_BADARG  # head_cap < 0
    assert lib.bmx_exchange_create(0, 0, 1, 0, 0, 0, 1, ctypes.byref(handle)) == E.BMX_E_BADARG   # depth < 2
    assert lib.bmx_exchange_create(-1, 0, 1, 0, 0, 0, 2, ctypes.byref(handle)) in either
    assert lib.bmx_scanner_create(0, None) == E.BMX_E_BADARG
    assert lib.bmx_scanner_create(-1, ctypes.byref(handle)) in either
    assert not handle.value


def test_no_cpu_fallback(bmx):
    """Without a CUDA device a scan must fail loudly, never quietly compute on the host."""
    if bmx.device_count() > 0:
        pytest.skip("a CUDA device is visible")
    with pytest.raises(bmx.BmxError) as e:
        bmx.search(b"hello world", b"o")
    assert e.value.code == bmx._lib.BMX_E_NODEVICE
    # m > n is still answered without a device only after the device check: no silent CPU path
    with pytest.raises(bmx.BmxError):
        bmx.search(b"ab", b"abc")
    with pytest.raises(bmx.BmxError) as e:
        bmx.find_first(b"hello world", b"o")
    assert e.value.code == bmx._lib.BMX_E_NODEVICE


def test_product_sources_never_touch_the_oracle():
    pkg = ROOT / "parallel_implementation_of_string_matching_algorithms_opencl_b200"
    for path in list(pkg.rglob("*.py")) + list(pkg.rglob("*.cu")) + list(pkg.rglob("*.cpp")) + list(pkg.rglob("*.h")):
        text = path.read_text()
        assert "liboracle" not in text and "libref_bm" not in text and "bm_oracle.h" not in text, path
