"""No search may see state or bytes left behind by an earlier call.

Between calls the library keeps results and buffers on the device and in pinned host memory: the host-mapped result
words of each thread's scanner (running count, find-first answer), the epoch-tagged find-first key word, the
self-cleaning scratch halves, the pattern cache, the thread's position list, its device copy of the last host text,
the pinned landing area of small host searches and host ranges, and the bounce buffers.  A test that repeats one
search cannot tell a stale result from a right one, so everything here is built so that the stale answer is wrong:

* a seeded call sequence over every entry point, in which each call's answer differs from the answers of the three
  calls before it and from the last call that wrote the same shared buffer (asserted on the CPU before anything
  runs), checked call by call, with device outputs in guard-banded buffers;
* text that ends inside an occurrence whose remaining bytes sit right behind it -- in the library's own buffer after
  a longer search, or in the caller's allocation around a device view;
* the find-first epoch counter wrapping after 65 000 searches of one thread;
* three threads running different sequences at once.

Truth is always computed on the exact bytes a call was given: the oracle (its multi-threaded form for large texts),
the KMP matcher for patterns beyond 2000 bytes, the lowered bytes for ignore_case, and per-range truth from the
whole-text list for ranges."""
from __future__ import annotations

import random
import threading
import zlib
from ctypes import byref, c_char_p, c_int32, c_int64, c_uint64, c_void_p
from dataclasses import dataclass

import numpy as np
import pytest

from test_exact_reference import kmp
from test_parity_gpu import _find_all, dev, to_dev  # noqa: F401  (dev is a fixture)
from test_paths_gpu import INSTANCES, set_knobs
from test_ranges_gpu import list_truth

torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu

SENT = 0x5A5A5A5A5A5A5A5A
G = 16                                          # sentinel entries on each side of a device output
LOWER = np.arange(256, dtype=np.uint8)
LOWER[65:91] += 32
EMPTY = np.zeros(0, dtype=np.int64)


def truth(oracle, text: np.ndarray, pat: bytes, ignore_case: bool = False) -> np.ndarray:
    """All occurrences of pat in exactly these bytes (ASCII case folded on both sides for ignore_case)."""
    text = np.ascontiguousarray(text, dtype=np.uint8)
    if ignore_case:
        text, pat = LOWER[text], pat.lower()
    if text.size < len(pat):
        return EMPTY
    if len(pat) > 2000:
        return kmp(oracle, text, pat)
    return oracle.search_np(text, pat) if text.size > (1 << 16) else oracle.search(text.tobytes(), pat)


def mixcase(pat: bytes, rnd: random.Random) -> bytes:
    return bytes(c ^ 0x20 if chr(c).isalpha() and chr(c).isascii() and rnd.random() < 0.5 else c for c in pat)


def variants_for(m: int):
    return ["auto", "window"] + (["qgram"] if m >= 7 else []) + (["shiftand"] if m <= 32 else [])


# ---------------------------------------------------------------------------------------------------------------
# The call-sequence generator (CPU)
# ---------------------------------------------------------------------------------------------------------------
BIG = 64 << 20
DENSE_AT, DENSE_LEN = 48 << 20, 6 << 20         # 'a'/'b' only: any two-byte pattern of them hits a quarter of starts
ALPHA = b"acgtACGT"
LEVELS = ((1, 300), (300, 1 << 16), (1 << 16, 4 << 20), (4 << 20, BIG))
SHAPE = (0, 1, 2, 3, 3, 2, 1, 0)                # text sizes rise to 64 MiB and fall back, so buffers grow, then get reused
KINDS = ("search", "search_device", "find_first", "find_first_device", "multi", "ranges", "partitions", "scanner")
WEIGHTS = (4, 4, 2, 2, 1.5, 1.5, 0.7, 1.3)
M_CHOICES = (1, 2, 3, 4, 5, 7, 8, 12, 16, 33, 64, 300, 2500)
LAYOUTS = ("default", "chunked", "ring")
LAYOUT_KNOBS = {"default": {}, "chunked": {"BMX_H2D_CHUNK_KB": "64"},
                "ring": {"BMX_RESIDENT_MAX_MB": "0", "BMX_H2D_CHUNK_KB": "64"}}
SMALL_HOST = 4 << 20                            # host texts up to this size take the one-stream path (bmx_host.cu)


@dataclass
class Call:
    kind: str
    text: np.ndarray                            # the exact bytes the call searches
    pat: object                                 # bytes, or a list of bytes (multi)
    cap: object                                 # None: room for all; 0: count only
    opt: dict
    want: object                                # the answer, in the entry point's own shape
    count: object = None                        # the total the call reports (None: find-first)
    first: object = None                        # the first position it returns (None: none returned)
    prefix: bytes = b""                         # the positions it returns
    writes: frozenset = frozenset()             # shared buffers the call writes: h_small, pos, key, scanner
    scan: str = ""                              # the thread's own scanner: count, positions or find scans
    room: int = 0                               # entries the thread's position list may hold after the call (upper bound)

    def tag(self):
        pats = [len(p) for p in self.pat] if isinstance(self.pat, list) else len(self.pat)
        return (self.kind, self.text.size, pats, self.cap, {k: v for k, v in self.opt.items() if k not in ("begin", "end", "se")})


def distinct(a: Call, b: Call) -> bool:
    """a's answer cannot be mistaken for b's, whatever the two entry points: another total (a search's count, a
    multi-pattern set's or a range set's sum of counts), another first returned position, another returned list.
    Fields one of the calls does not report (find-first: no total; count-only: no positions) are not compared."""
    if a.count is not None and a.count == b.count:
        return False
    if a.first is not None and a.first == b.first:
        return False
    return not (a.prefix and a.prefix == b.prefix)


def base_text(seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    text = np.frombuffer(ALPHA, dtype=np.uint8)[rng.integers(0, len(ALPHA), BIG, dtype=np.uint8)]
    text[DENSE_AT:DENSE_AT + DENSE_LEN] = np.frombuffer(b"ab", dtype=np.uint8)[rng.integers(0, 2, DENSE_LEN, dtype=np.uint8)]
    return text


def pick_cap(rnd: random.Random, count: int, host: bool):
    """None (room for all), 1, a cut inside the list, or more than the count."""
    kind = rnd.choice(("all", "one", "inside", "above"))
    if kind == "all":
        return None if host else max(count, 1)
    if kind == "one":
        return 1
    if kind == "inside" and count >= 3:
        return rnd.randint(2, count - 1)
    return count + rnd.randint(1, 5)


def held(full: np.ndarray, cap) -> np.ndarray:
    return full if cap is None else full[:cap]


def draw_pattern(rnd: random.Random, text: np.ndarray, m: int) -> bytes:
    if text.size >= m and rnd.random() < 0.75:
        o = rnd.randrange(0, text.size - m + 1)
        return text[o:o + m].tobytes()
    pat = bytearray(rnd.choice(ALPHA) for _ in range(m))
    if rnd.random() < 0.5:
        pat[rnd.randrange(m)] = ord("z")                      # occurs nowhere
    return bytes(pat)


def first_room(n: int, count: int) -> int:
    """An upper bound of the entries a search that writes the thread's position list leaves it with: the first guess
    max(2^20, n / 64) or the count, in whole MiB (bmx_ctx.h: first_pos_cap, ensure_buf)."""
    return -(-max(1 << 20, n // 64, count) * 8 // (1 << 20)) * (1 << 20) // 8


def draw_call(oracle, rnd: random.Random, base: np.ndarray, i: int, ncalls: int, knobs: bool, dense) -> Call:
    """One call of the sequence.  dense: None, or a call over the 'a'/'b' stretch with more than 2^20 hits: "search" or
    "ranges" (5-6 MiB), or "small" (a host search of at most 4 MiB for one byte, about 2 M hits: more than the first
    position buffer of the small-text path, which then scans its resident copy again)."""
    kind = "search" if dense == "small" else dense or rnd.choices(KINDS, WEIGHTS)[0]
    level = SHAPE[i * len(SHAPE) // ncalls]
    if rnd.random() < 0.35:
        level = rnd.randint(0, level)
    lo, hi = LEVELS[level]
    n = rnd.randrange(lo, hi)
    layout = rnd.choice(LAYOUTS) if knobs and kind in ("search", "find_first", "multi", "ranges", "partitions") else "default"
    if layout != "default" or kind == "partitions":
        n = min(n, 8 << 20)                    # 64 KiB chunks: keep the number of chunks in the hundreds
    if dense == "small":
        layout = "default"
        n = rnd.randrange(SMALL_HOST - (1 << 19), SMALL_HOST + 1)
        off = DENSE_AT + rnd.randrange(0, DENSE_LEN - n)
        pat = rnd.choice((b"a", b"b"))
    elif dense:
        n = rnd.randrange(5 << 20, DENSE_LEN)
        off = DENSE_AT + rnd.randrange(0, DENSE_LEN - n)
        pat = rnd.choice((b"ab", b"ba", b"aa", b"bb"))
    else:
        off = rnd.randrange(0, BIG - n + 1)
        m = rnd.choice([x for x in M_CHOICES if level < 3 or x >= 5])
        pat = draw_pattern(rnd, base[off:off + n], m)
    text = base[off:off + n]
    m = len(pat)
    opt = {"layout": layout, "pinned": rnd.random() < 0.4}
    ic = kind in ("search", "search_device", "scanner") and not dense and rnd.random() < 0.3
    if ic:
        pat = mixcase(pat, rnd)
        opt["ignore_case"] = True
    full = truth(oracle, text, pat, ic)
    c = Call(kind, text, pat, None, opt, None)

    if kind in ("search", "search_device", "scanner"):
        c.cap = None if dense else (0 if rnd.random() < 0.4 else pick_cap(rnd, full.size, kind == "search"))
        out = held(full, c.cap)
        if kind == "search":
            c.want = (full.size, out)
            small = layout == "default" and n <= SMALL_HOST
            if c.cap != 0:
                c.writes = frozenset({"pos", "h_small"} if small else {"pos"})
                c.room = first_room(n, full.size)
        else:
            opt["variant"] = rnd.choice(variants_for(m))
            base_pos = rnd.choice((0, 0, 12345, (1 << 40) + 7))
            opt["pos_base"] = base_pos
            opt["stream"] = rnd.choice((None, 0, 1))
            if kind == "scanner":
                opt["head"] = rnd.choice((0, 1, 7, 100))
                k = rnd.choice((1, 1, 2, 3))
                opt["cuts"] = sorted(rnd.randint(0, n) for _ in range(k - 1))
                c.writes = frozenset({"scanner"})      # a Scanner object of its own, not the thread's
            out = out + base_pos
            c.want = (full.size, out)
        c.count, c.first, c.prefix = full.size, (int(out[0]) if out.size else None), out.tobytes()
        if kind != "scanner":
            c.scan = "count" if c.cap == 0 else "positions"
    elif kind in ("find_first", "find_first_device"):
        opt["stream"] = rnd.choice((None, 0, 1))
        c.want = int(full[0]) if full.size else -1
        c.first = c.want
        c.writes = frozenset({"key"})
        c.scan = "find"
    elif kind == "multi":
        host = rnd.random() < 0.5
        eligible = rnd.random() < 0.6
        k = rnd.randint(2, 5)
        ms = [rnd.choice((7, 8, 12, 16, 33, 300)) for _ in range(k)] if eligible else [rnd.choice((2, 3, 5, 9)) for _ in range(k)]
        pats = [draw_pattern(rnd, text, mm) for mm in ms]
        fulls = [truth(oracle, text, p) for p in pats]
        top = max(f.size for f in fulls)
        c.pat = pats
        c.cap = 0 if rnd.random() < 0.3 else pick_cap(rnd, top, host)
        opt.update(host=host, stream=rnd.choice((None, 0, 1)))
        outs = [held(f, c.cap) for f in fulls]
        c.want = [(f.size, o) for f, o in zip(fulls, outs)]
        c.count = sum(f.size for f in fulls)
        ret = [o for o in outs if o.size]
        c.first = int(ret[0][0]) if ret else None
        c.prefix = b"".join(o.tobytes() for o in outs)
        if c.cap != 0:                         # the union list of one pass, or one pattern after another
            c.writes = frozenset({"pos"})
            c.room = first_room(n, c.count)
    elif kind == "ranges":
        host = rnd.random() < 0.5
        d = rnd.randint(1, 40)
        begin, end = [], []
        for j in range(d):
            a = rnd.choice((0, rnd.randrange(0, n + 1), max(0, n - rnd.randint(0, 3 * m))))
            b = rnd.choice((n, min(n, a + rnd.randint(0, 3 * m)), rnd.randint(a, n)))
            begin.append(a)
            end.append(b)
        begin[0], end[-1] = 0, n                                        # ranges touching both ends of the text
        if dense:
            end[0] = n
        counts, offsets, pos = list_truth(full, m, begin, end)
        total = int(offsets[-1])
        c.cap = None if dense and host else (0 if rnd.random() < 0.25 else pick_cap(rnd, total, host))
        opt.update(host=host, begin=begin, end=end, stream=rnd.choice((None, 0, 1)))
        out = held(pos, c.cap)
        c.want = (counts, offsets, out)
        c.count = total
        c.first = int(out[0]) if out.size else None
        c.prefix = out.tobytes()
        c.writes = frozenset({"pos", "h_small"})
        c.scan = "positions"
        c.room = first_room(n, full.size)
    elif kind == "partitions":
        se = []
        for _ in range(rnd.randint(1, 12)):
            a = rnd.randrange(0, n)
            se += [a, rnd.choice((n - 1, rnd.randint(a - 1, n - 1), min(n - 1, a + 2 * m)))]
        se = np.array(se, dtype=np.int32)
        b = se[0::2].astype(np.int64)
        e = np.maximum(se[1::2].astype(np.int64) + 1, b)
        counts, _, _ = list_truth(full, m, b, e)
        opt["se"] = se
        c.want = counts.astype(np.int32)
        c.count = int(counts.sum())
        c.writes = frozenset({"pos", "h_small"})
        c.scan = "positions"
        c.room = first_room(n, full.size)
    return c


def make_calls(oracle, seed: int, ncalls: int = 150, knobs: bool = True) -> list[Call]:
    """ncalls calls in which each answer differs from the three before it and from the last call that wrote any
    shared buffer it writes.  The rule is asserted here, before anything runs."""
    rnd = random.Random(seed)
    base = base_text(seed)
    calls, last = [], {}
    dense_at = {10: "small", ncalls // 4: "search", ncalls // 2 + 3: "ranges", 3 * ncalls // 4: "search"}
    ndev = 0
    for i in range(ncalls):
        dense = dense_at.get(i) or (rnd.choice(("search", "ranges")) if i > 10 and rnd.random() < 0.02 else None)
        for _attempt in range(200):
            c = draw_call(oracle, rnd, base, i, ncalls, knobs, dense)
            others = calls[-3:] + [last[b] for b in c.writes if b in last]
            if all(distinct(c, o) for o in others):
                break
        for o in calls[-3:] + [last[b] for b in c.writes if b in last]:
            assert distinct(c, o), (seed, i, c.tag(), o.tag())
        if c.kind in ("search_device", "find_first_device", "scanner") or (c.kind in ("multi", "ranges") and not c.opt["host"]):
            c.opt["misalign"] = ndev % 16                               # device text starts misalign bytes past a 16-byte boundary
            ndev += 1
        calls.append(c)
        for b in c.writes:
            last[b] = c
    return calls


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_call_generator_distinct_and_covering(oracle, seed):
    """CPU: the sequence obeys the distinctness rule (make_calls asserts it) and reaches what the GPU tests rely on:
    every entry point, layout and source, misalignments 0..15, every cap class, text sizes up to 64 MiB and back down,
    dense calls past the first 2^20-entry position buffer (one of them a small host text denser than any position list
    the calls before it can have left), and every transition between count-only, positions and find-first scans on
    directly consecutive calls that use the thread's own scanner."""
    calls = make_calls(oracle, seed)
    assert {c.kind for c in calls} == set(KINDS)
    host = [c for c in calls if c.kind in ("search", "find_first") or (c.kind in ("multi", "ranges") and c.opt["host"])]
    assert {(c.opt["layout"], c.opt["pinned"]) for c in host} >= {(lay, p) for lay in LAYOUTS for p in (False, True)}
    assert any(c.kind == "search" and c.opt["layout"] == "default" and 0 < c.text.size <= SMALL_HOST and c.cap != 0 for c in calls)
    assert {c.opt["misalign"] for c in calls if "misalign" in c.opt} == set(range(16))
    dev_calls = [c for c in calls if c.kind == "search_device"]
    assert {c.opt["stream"] for c in dev_calls} == {None, 0, 1} and any(c.opt.get("ignore_case") for c in dev_calls)
    assert any(c.opt["pos_base"] for c in dev_calls) and len({c.opt["variant"] for c in dev_calls}) >= 3
    multi = {(c.opt["host"], all(7 <= len(p) for p in c.pat)) for c in calls if c.kind == "multi"}
    assert len(multi) >= 3
    caps = set()
    for c in calls:
        if c.kind in ("search", "search_device", "scanner", "ranges", "multi"):
            total = max(w[0] for w in c.want) if c.kind == "multi" else c.count
            caps.add("none" if c.cap is None else "zero" if c.cap == 0 else "one" if c.cap == 1 else
                     "inside" if c.cap < total else "above")
    assert caps == {"none", "zero", "one", "inside", "above"}
    sizes = [c.text.size for c in calls]
    top = int(np.argmax(sizes))
    assert sizes[top] > (32 << 20) and min(sizes[top:]) < 300 and min(sizes[:top]) < 300
    assert any(c.cap is None and c.kind in ("search", "ranges") and c.want[-1].size > (1 << 20) for c in calls)
    rescans = [i for i, c in enumerate(calls) if c.kind == "search" and c.opt["layout"] == "default" and c.cap is None and
               c.text.size <= SMALL_HOST and c.count > max([1 << 20] + [p.room for p in calls[:i]])]
    assert rescans, "no small host text denser than the position list the calls before it may have left"
    scans = [c.scan for c in calls]
    pairs = {(a, b) for a, b in zip(scans, scans[1:]) if a and b}
    assert pairs == {(a, b) for a in ("count", "positions", "find") for b in ("count", "positions", "find")}


def test_truth_helpers(oracle):
    """CPU: the truth used above against a brute-force scan, ignore_case folding only ASCII letters."""
    rnd = random.Random(5)
    for _ in range(200):
        n = rnd.randint(0, 300)
        text = np.frombuffer(bytes(rnd.choice(b"aAbB@[`{\xc1\xe1") for _ in range(n)), dtype=np.uint8)
        pat = bytes(rnd.choice(b"aAbB@[`{\xc1\xe1") for _ in range(rnd.randint(1, 4)))
        for ic in (False, True):
            t, p = (bytes(text).lower(), pat.lower()) if ic else (bytes(text), pat)
            want = [i for i in range(len(t) - len(p) + 1) if t[i:i + len(p)] == p]
            assert list(truth(oracle, text, pat, ic)) == want
    big = np.frombuffer(b"ab" * 3000, dtype=np.uint8)
    assert np.array_equal(truth(oracle, big, b"ab" * 1100), _find_all(big.tobytes(), b"ab" * 1100))   # the KMP branch
    counts, offsets, pos = list_truth(truth(oracle, big, b"aba"), 3, [0, 5, 10], [5, 10, 10])
    assert list(counts) == [2, 1, 0] and list(offsets) == [0, 2, 3, 3] and list(pos) == [0, 2, 1]


def test_scanner_rejects_host_and_wrongly_typed_tensors(bmx):
    """CPU: Scanner.scan / begin / export_result take raw device pointers, so a CPU tensor is refused before the
    library sees its address."""
    sc = object.__new__(bmx.Scanner)            # no device: the checks come before any library call
    sc._lib, sc._h = bmx._lib.load(), c_void_p()
    with pytest.raises(TypeError):
        sc.scan(torch.zeros(64, dtype=torch.uint8))
    with pytest.raises(TypeError):
        sc.scan(np.zeros(64, dtype=np.uint8))
    with pytest.raises(TypeError):
        sc.begin(torch.zeros(8, dtype=torch.int64))
    with pytest.raises(TypeError):
        sc.export_result(torch.zeros(8, dtype=torch.int64))


# ---------------------------------------------------------------------------------------------------------------
# Running a call (GPU)
# ---------------------------------------------------------------------------------------------------------------
def guarded(k: int, device):
    return torch.full((k + 2 * G,), SENT, dtype=torch.int64, device=device)


def assert_guarded(buf, out: np.ndarray, tag):
    """buf holds out at [G, G + len(out)) and the sentinel everywhere else."""
    got = buf.cpu().numpy()
    want = np.full(got.size, SENT, dtype=np.int64)
    want[G:G + out.size] = out
    if not np.array_equal(got, want):
        bad = np.flatnonzero(got != want)
        raise AssertionError(f"{tag}: {bad.size} entries differ, first at {int(bad[0]) - G} (G = {G}): "
                             f"got {int(got[bad[0]]):#x}, want {int(want[bad[0]]):#x}")


def host_source(text: np.ndarray, pinned: bool):
    return torch.from_numpy(text.copy()).pin_memory() if pinned else text


class Runner:
    """Runs calls of one sequence on the calling thread, each checked in full against its answer."""

    def __init__(self, bmx, device, streams, scanner, monkeypatch=None, mg=None):
        self.bmx, self.lib, self.dev = bmx, bmx._lib.load(), device
        self.streams, self.scanner, self.mp, self.mg = streams, scanner, monkeypatch, mg

    def stream(self, c: Call):
        """The call's stream, made to wait for everything enqueued so far on the current stream: call it after the
        inputs are copied and the guard bands filled, right before the library call."""
        st = None if c.opt.get("stream") is None else self.streams[c.opt["stream"]]
        if st is not None:
            st.wait_stream(torch.cuda.current_stream(self.dev))   # inputs made on the current stream
        return st

    def handle(self, st):
        return (st or torch.cuda.current_stream(self.dev)).cuda_stream

    def run(self, c: Call, tag):
        tag = (*tag, *c.tag())
        if self.mp is not None:
            for k in ("BMX_H2D_CHUNK_KB", "BMX_RESIDENT_MAX_MB"):
                self.mp.delenv(k, raising=False)
            for k, v in LAYOUT_KNOBS[c.opt["layout"]].items():
                self.mp.setenv(k, v)
        getattr(self, "run_" + c.kind)(c, tag)

    def device_text(self, c: Call):
        return to_dev(c.text, self.dev, misalign=c.opt["misalign"])

    def run_search(self, c, tag):
        src = host_source(c.text, c.opt["pinned"])
        count, pos = self.bmx.search(src, c.pat, max_positions=c.cap, ignore_case=c.opt.get("ignore_case", False))
        assert count == c.want[0] and np.array_equal(pos, c.want[1]), (*tag, count, pos.size)
        if self.mg is not None and not c.opt.get("ignore_case"):
            count, pos, _ = self.mg.search(src, c.pat, max_positions=c.cap)
            assert count == c.want[0] and np.array_equal(pos, c.want[1]), (*tag, "multi-GPU")

    def run_search_device(self, c, tag):
        td = self.device_text(c)
        buf = guarded(c.cap, self.dev) if c.cap else None
        st = self.stream(c)                                     # after every input and guard fill is enqueued
        count, _, _ = self.bmx.search_device(td, c.pat, pos_out=None if buf is None else buf[G:G + c.cap],
                                             pos_base=c.opt["pos_base"], variant=c.opt["variant"], stream=st, timing=False,
                                             ignore_case=c.opt.get("ignore_case", False))
        assert count == c.want[0], (*tag, count)
        if buf is not None:
            assert_guarded(buf, c.want[1], tag)

    def run_find_first(self, c, tag):
        got = self.bmx.find_first(host_source(c.text, c.opt["pinned"]), c.pat)
        assert got == c.want, (*tag, got)

    def run_find_first_device(self, c, tag):
        td = self.device_text(c)
        got = self.bmx.find_first_device(td, c.pat, stream=self.stream(c))
        assert got == c.want, (*tag, got)

    def run_multi(self, c, tag):
        if c.opt["host"]:
            got = self.bmx.search_multi(host_source(c.text, c.opt["pinned"]), c.pat, max_positions=c.cap)
            for k, ((count, pos), (wc, wp)) in enumerate(zip(got, c.want)):
                assert count == wc and np.array_equal(pos, wp), (*tag, k, count, pos.size)
            return
        td = self.device_text(c)
        k, cap = len(c.pat), c.cap
        bufs = [guarded(cap, self.dev) for _ in c.pat] if cap else []
        st = self.stream(c)
        counts = (c_uint64 * k)()
        self.bmx._lib.check(self.lib.bmx_search_multi_device(
            c_void_p(td.data_ptr() if td.numel() else 0), td.numel(), k, (c_char_p * k)(*c.pat),
            (c_int32 * k)(*[len(p) for p in c.pat]), (c_void_p * k)(*[b.data_ptr() + 8 * G for b in bufs] if cap else [None] * k),
            (c_int64 * k)(*[cap] * k), counts, c_void_p(self.handle(st))))
        for j, (wc, wp) in enumerate(c.want):
            assert int(counts[j]) == wc, (*tag, j, int(counts[j]))
            if cap:
                assert_guarded(bufs[j], wp, (*tag, j))

    def run_ranges(self, c, tag):
        begin = np.array(c.opt["begin"], dtype=np.int64)
        end = np.array(c.opt["end"], dtype=np.int64)
        wc, wo, wp = c.want
        if c.opt["host"]:
            counts, offsets, pos = self.bmx.search_ranges(host_source(c.text, c.opt["pinned"]), c.pat, begin, end,
                                                          max_positions=c.cap)
            assert np.array_equal(counts, wc) and np.array_equal(offsets, wo), (*tag, "counts")
            assert np.array_equal(pos, wp), (*tag, "positions", pos.size)
            return
        td = self.device_text(c)
        d, cap = begin.size, c.cap
        bd = torch.from_numpy(begin).to(self.dev)
        ed = torch.from_numpy(end).to(self.dev)
        counts = torch.full((d + 1,), -1, dtype=torch.int64, device=self.dev)
        offsets = torch.full((d + 2,), -1, dtype=torch.int64, device=self.dev)
        buf = guarded(cap, self.dev) if cap else None
        st = self.stream(c)
        total = c_uint64()
        self.bmx._lib.check(self.lib.bmx_search_ranges_device(
            c_void_p(td.data_ptr() if td.numel() else 0), td.numel(), d, c_void_p(bd.data_ptr()), c_void_p(ed.data_ptr()),
            c.pat, len(c.pat), c_void_p(buf.data_ptr() + 8 * G) if cap else None, cap or 0, c_void_p(counts.data_ptr()),
            c_void_p(offsets.data_ptr()), byref(total), c_void_p(self.handle(st))))
        assert total.value == int(wo[-1]), (*tag, "total", total.value)
        got_c, got_o = counts.cpu().numpy(), offsets.cpu().numpy()
        assert np.array_equal(got_c[:d], wc.astype(np.int64)) and got_c[d] == -1, (*tag, "counts")
        assert np.array_equal(got_o[:d + 1], wo) and got_o[d + 1] == -1, (*tag, "offsets")
        if buf is not None:
            assert_guarded(buf, wp, tag)

    def run_partitions(self, c, tag):
        src = host_source(c.text, c.opt["pinned"])
        got = self.bmx.search_partitions(src, c.pat, c.opt["se"])
        assert np.array_equal(got, c.want), (*tag, got, c.want)

    def run_scanner(self, c, tag):
        td = self.device_text(c)
        sc, n, m, cap = self.scanner, c.text.size, len(c.pat), c.cap
        buf = guarded(cap, self.dev) if cap else None
        head = c.opt["head"]
        packed = guarded(head + 2, self.dev)
        st = self.stream(c)
        h = self.handle(st)
        sc.set_pattern(c.pat, variant=c.opt["variant"], stream=h, ignore_case=c.opt.get("ignore_case", False))
        sc.begin(None if buf is None else buf[G:G + cap], stream=h)
        lo = 0
        for cut in c.opt["cuts"] + [n]:
            hi = cut if cut == n else min(n, cut + m - 1)       # the piece holding the starts [lo, cut)
            if hi - lo >= m:
                sc.scan(td[lo:hi], c.opt["pos_base"] + lo, stream=h)
            lo = max(lo, cut)
        sc.export_result(packed[G:G + head + 2], stream=h)
        count, _ = sc.finish(stream=h)
        wc, wp = c.want
        assert count == wc, (*tag, count)
        if buf is not None:
            assert_guarded(buf, wp, tag)
        k = wp.size if cap else 0
        assert_guarded(packed, np.concatenate([[wc, k], wp[:min(head, k)]]).astype(np.int64), (*tag, "export"))


def run_sequence(runner: Runner, calls, tag):
    for i, c in enumerate(calls):
        runner.run(c, (*tag, i))


@gpu
def test_interleaved_entry_points(bmx, oracle, dev, monkeypatch):  # noqa: F811
    """3 seeds x 150 calls over every entry point on one host thread, each call's answer different from the answers
    its shared state last held; every call checked in full."""
    streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
    mg = bmx.MultiGpu(0) if bmx.device_count() >= 2 else None
    sc = bmx.Scanner(0)
    try:
        runner = Runner(bmx, dev, streams, sc, monkeypatch, mg)
        for seed in (1, 2, 3):
            run_sequence(runner, make_calls(oracle, seed), ("seed", seed))
    finally:
        sc.close()
        if mg is not None:
            mg.close()


@gpu
def test_threads_run_distinct_sequences_at_once(bmx, oracle, dev):  # noqa: F811
    """3 host threads, each with its own seed, stream pair and scanner, run different call sequences at the same time:
    no thread may read another's results or buffers.  (Layout knobs are process-wide, so every host call here takes the
    default layout.)"""
    seqs = [make_calls(oracle, seed, ncalls=60, knobs=False) for seed in (11, 12, 13)]
    errors = []
    start = threading.Barrier(len(seqs))

    def work(t, calls):
        try:
            torch.cuda.set_device(dev)
            sc = bmx.Scanner(0)
            runner = Runner(bmx, dev, [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)], sc)
            start.wait()
            run_sequence(runner, calls, ("thread", t))
            sc.close()
        except BaseException as e:  # noqa: BLE001
            errors.append((t, repr(e)[:2000]))

    threads = [threading.Thread(target=work, args=(t, calls)) for t, calls in enumerate(seqs)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors


# ---------------------------------------------------------------------------------------------------------------
# Bytes behind the text: the library's buffers after a longer search
# ---------------------------------------------------------------------------------------------------------------
STALE_MS = (1, 2, 3, 4, 5, 7, 16, 33, 64, 1025, 5000)
CHUNK = 64 << 10


@gpu
@pytest.mark.parametrize("layout", ["small", "chunked", "ring"])
def test_stale_bytes_behind_the_text(bmx, oracle, monkeypatch, layout):
    """Search T, then T[:n2] with n2 inside T's only occurrence: the library's copy of the text still holds T's bytes
    behind n2, and they complete the occurrence.  Neither search, count-only search, search_multi, find_first nor a host
    range that ends at n2 may report it.  ignore_case runs have the bytes behind n2 in the opposite case."""
    set_knobs(monkeypatch, **({} if layout == "small" else LAYOUT_KNOBS[layout]))
    rng = np.random.default_rng(zlib.crc32(layout.encode()))
    digits = np.frombuffer(b"0123456789", dtype=np.uint8)
    N = 5 * CHUNK + 4321
    for m in STALE_MS:
        cuts = sorted({m - 1, max(m // 2, 1), 1} - {m}) if m > 1 else [0]   # bytes of the occurrence in front of n2
        for ic in (False, True):
            pat_arr = rng.integers(97, 123, size=m, dtype=np.uint8)
            pat = pat_arr.tobytes()
            other = rng.integers(97, 123, size=max(m, 7), dtype=np.uint8).tobytes()
            for cut in cuts:
                n2 = 3 * CHUNK + 777 + int(rng.integers(0, 5000))
                q = n2 - cut
                T = digits[rng.integers(0, 10, size=max(N, q + m + 10))]
                T[q:q + m] = pat_arr
                if ic:
                    T[n2:q + m] -= 32                                    # the bytes behind n2 in upper case
                head = T[:n2]
                want_T, want_h = truth(oracle, T, pat, ic), truth(oracle, head, pat, ic)
                assert list(want_T) == [q] and want_h.size == 0
                for pinned in (False, True):
                    tag = (layout, m, ic, cut, pinned)
                    src_T, src_h = host_source(T, pinned), host_source(head, pinned)
                    count, pos = bmx.search(src_T, pat, ignore_case=ic)
                    assert count == 1 and list(pos) == [q], tag
                    count, pos = bmx.search(src_h, pat, ignore_case=ic)
                    assert count == 0 and pos.size == 0, (*tag, "search", list(pos[:4]))
                    count, _ = bmx.search(src_h, pat, max_positions=0, ignore_case=ic)
                    assert count == 0, (*tag, "count-only")
                    if ic:
                        continue
                    got = bmx.search_multi(src_T, [pat, other])
                    assert got[0][0] == 1, (*tag, "multi T")
                    got = bmx.search_multi(src_h, [pat, other])
                    wants = [want_h, truth(oracle, head, other)]
                    for (count, pos), w in zip(got, wants):
                        assert count == w.size and np.array_equal(pos, w), (*tag, "multi")
                    begin, end = [0, max(0, n2 - 3 * m), n2], [n2, n2, T.size]
                    counts, offsets, pos = bmx.search_ranges(src_T, pat, begin, end)
                    wc, wo, wp = list_truth(want_T, m, begin, end)
                    assert wc[0] == wc[1] == 0 and np.array_equal(counts, wc), (*tag, "ranges", list(counts))
                    assert np.array_equal(offsets, wo) and np.array_equal(pos, wp), (*tag, "ranges")
                    assert bmx.find_first(src_T, pat) == q
                    assert bmx.find_first(src_h, pat) == -1, (*tag, "find_first")


# ---------------------------------------------------------------------------------------------------------------
# Bytes around a device view: the caller's allocation in front of and behind the text
# ---------------------------------------------------------------------------------------------------------------
def poisoned_view(rng, pat: np.ndarray, poison: np.ndarray, n: int, mis: int, plant: np.ndarray | None, dev):  # noqa: F811
    """buf[off:off + n] with off % 16 == mis.  In front of the view the poison bytes start an occurrence that the view's
    first bytes finish (k of its bytes outside, k = m: a whole occurrence right in front); behind it the view's last j
    bytes start one that the poison bytes finish.  The scan fetches the text from the 16-byte boundary below the view,
    so with mis > 0 the front occurrence starts inside the fetched bytes (k <= mis): only the masking of starts in
    front of the view keeps it out.  (With mis = 0 nothing in front of the view is fetched.)"""
    m = pat.size
    if mis == 0:
        k = 1
    else:
        k = min(m, mis) if mis % 2 else 1 + (mis // 2) % min(m, mis)
    j = (m - 1) - mis % m
    off = 64 + mis
    full = np.frombuffer(b"0123456789", dtype=np.uint8)[rng.integers(0, 10, size=off + n + m + 64)]
    view = full[off:off + n]
    if plant is not None:
        for s in (n // 3, n // 2 + 1):
            view[s:s + m] = plant
    full[off - k:off] = poison[:k]
    view[:m - k] = pat[k:]
    view[n - j:] = pat[:j]
    full[off + n:off + n + m - j] = poison[j:]
    buf = torch.from_numpy(full).to(dev)
    return view.copy(), buf[off:off + n]


@gpu
@pytest.mark.parametrize("label,variant,m,ndistinct,knobs", INSTANCES, ids=[i[0] for i in INSTANCES])
def test_poisoned_surroundings_of_device_views(bmx, oracle, dev, monkeypatch, label, variant, m, ndistinct, knobs):  # noqa: F811
    """Every filter kind, exact and folded, misalignments 0..15 and both tile sizes: the bytes in front of the view
    complete a match with its head and the bytes behind complete one with its tail.  Count-only, positions with
    pos_base, find_first_device, search_multi_device and search_ranges_device with ranges touching 0 and n see the
    view's own matches only (odd misalignments: none at all)."""
    lib = bmx._lib.load()
    rng = np.random.default_rng(zlib.crc32(label.encode()) + 7)
    unit = rng.choice(np.arange(97, 123, dtype=np.uint8), size=ndistinct, replace=False)
    pat_arr = np.resize(unit, m)
    pat = pat_arr.tobytes()
    other = pat_arr[::-1].copy()
    other[0] = ord("q") if other[0] != ord("q") else ord("r")
    n = 20_000 + 3 * m
    set_knobs(monkeypatch, **knobs)
    for ic in (False, True):
        poison = pat_arr - 32 if ic else pat_arr                        # folded runs: the outside bytes in upper case
        for mis in range(16):
            plant = None if mis % 2 else (np.where(rng.random(m) < 0.5, pat_arr - 32, pat_arr).astype(np.uint8) if ic else pat_arr)
            host, td = poisoned_view(rng, pat_arr, poison, n, mis, plant, dev)
            want = truth(oracle, host, pat, ic)
            assert want.size == (0 if mis % 2 else 2), (label, ic, mis, want)
            base = 0 if mis % 4 == 0 else (1 << 40) + mis
            for tile in (16384, 32768):
                tag = (label, ic, mis, tile)
                set_knobs(monkeypatch, BMX_TILE=tile)
                count, _, _ = bmx.search_device(td, pat, variant=variant, timing=False, ignore_case=ic)
                assert count == want.size, (*tag, "count-only", count)
                buf = guarded(want.size + 2, dev)
                count, _, stats = bmx.search_device(td, pat, pos_out=buf[G:G + want.size + 2], pos_base=base, variant=variant,
                                                    ignore_case=ic)
                assert count == want.size and stats["tile_bytes"] == tile, (*tag, "positions", count)
                assert_guarded(buf, want + base, (*tag, "positions"))
                if ic:
                    continue
                assert bmx.find_first_device(td, pat) == (int(want[0]) if want.size else -1), (*tag, "find_first")
                pats = [pat, other.tobytes()]
                wants = [want, truth(oracle, host, pats[1])]
                bufs = [guarded(4, dev) for _ in pats]
                counts = (c_uint64 * 2)()
                bmx._lib.check(lib.bmx_search_multi_device(c_void_p(td.data_ptr()), n, 2, (c_char_p * 2)(*pats),
                                                           (c_int32 * 2)(m, m), (c_void_p * 2)(*[b.data_ptr() + 8 * G for b in bufs]),
                                                           (c_int64 * 2)(4, 4), counts, c_void_p(torch.cuda.current_stream().cuda_stream)))
                for k in range(2):
                    assert int(counts[k]) == wants[k].size, (*tag, "multi", k, int(counts[k]))
                    assert_guarded(bufs[k], wants[k][:4], (*tag, "multi", k))
                begin = [0, 0, n - m, n - m - 5, n // 4, n]
                end = [n, m + 5, n, n, n // 2 + m + 3, n]
                counts, offsets, pos = list_truth(want, m, begin, end)
                c_, o_, p_ = bmx.search_ranges_device(td, pat, torch.tensor(begin, device=dev), torch.tensor(end, device=dev),
                                                      max_positions=int(offsets[-1]) + 1)
                assert np.array_equal(c_.cpu().numpy(), counts.astype(np.int64)), (*tag, "ranges", c_.cpu().numpy())
                assert np.array_equal(o_.cpu().numpy(), offsets) and np.array_equal(p_.cpu().numpy(), pos), (*tag, "ranges")


# ---------------------------------------------------------------------------------------------------------------
# The find-first epoch wrap
# ---------------------------------------------------------------------------------------------------------------
WRAP = 65_000                                  # find-first searches of one scanner before its key word is cleared


@gpu
def test_find_first_epoch_wrap(bmx, dev):  # noqa: F811
    """A fresh thread (a fresh context: epoch counter 0) makes WRAP + 200 find-first searches whose answers cycle
    through an early position, a late one and -1; the search that ends the epoch range finds a match, so its key word
    outranks every later epoch unless the wrap clears it.  Around the wrap, host find_first and count-only
    search_device calls are interleaved."""
    lib = bmx._lib.load()
    W, m = 4096, 9
    pat = b"needle\x01\x02\x03"[:m]
    texts = [np.frombuffer(b"0123456789", dtype=np.uint8)[np.random.default_rng(k).integers(0, 10, W)] for k in range(3)]
    texts[0][100:100 + m] = np.frombuffer(pat, dtype=np.uint8)            # early
    texts[1][3000:3000 + m] = np.frombuffer(pat, dtype=np.uint8)          # late
    answers = [100, 3000, -1]
    counts = [1, 1, 0]
    td = torch.from_numpy(np.concatenate(texts)).to(dev)
    torch.cuda.synchronize()
    ptrs = [c_void_p(td.data_ptr() + k * W) for k in range(3)]
    assert (WRAP - 1) % 3 == 1                                            # the last search before the wrap: a late match
    out, errors = [], []

    def work():
        try:
            first = c_int64()
            ref = byref(first)
            fn = lib.bmx_find_first_device
            stream = c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            for i in range(WRAP + 200):
                k = i % 3
                if WRAP - 10 <= i < WRAP + 10:
                    if i % 2:
                        got = bmx.find_first(texts[k], pat)
                    else:
                        rc = fn(ptrs[k], W, pat, m, ref, stream)
                        got = first.value if rc == 0 else ("rc", rc)
                    c, _, _ = bmx.search_device(td[k * W:(k + 1) * W], pat, timing=False)
                    if c != counts[k]:
                        out.append((i, "count-only", c))
                else:
                    rc = fn(ptrs[k], W, pat, m, ref, stream)
                    got = first.value if rc == 0 else ("rc", rc)
                if got != answers[k]:
                    out.append((i, got, answers[k]))
                    if len(out) > 20:
                        break
        except BaseException as e:  # noqa: BLE001
            errors.append(repr(e))

    t = threading.Thread(target=work)
    t.start()
    t.join()
    assert not errors, errors
    assert not out, out[:20]


# ---------------------------------------------------------------------------------------------------------------
# Scanner argument checks on the device
# ---------------------------------------------------------------------------------------------------------------
@gpu
def test_scanner_rejects_strided_views(bmx, oracle, dev):  # noqa: F811
    """td[::2] is a CUDA uint8 tensor whose data_ptr() walks other bytes: Scanner.scan refuses it, as search_device
    does, and the scanner still searches a proper tensor afterwards."""
    text = np.frombuffer(b"xaxbxaxbxcab" * 1000, dtype=np.uint8)
    td = to_dev(text, dev)
    sc = bmx.Scanner(0)
    try:
        sc.set_pattern(b"ab")
        with pytest.raises(TypeError):
            sc.scan(td[::2])
        with pytest.raises(TypeError):
            sc.begin(torch.empty(8, dtype=torch.int32, device=dev))
        with pytest.raises(TypeError):
            sc.begin(torch.empty(16, dtype=torch.int64, device=dev)[::2])
        with pytest.raises(TypeError):
            sc.export_result(torch.empty(8, dtype=torch.int64))
        want = truth(oracle, text, b"ab")
        out = torch.empty(want.size, dtype=torch.int64, device=dev)
        sc.begin(out)
        sc.scan(td)
        count, _ = sc.finish()
        assert count == want.size and np.array_equal(out.cpu().numpy(), want)
    finally:
        sc.close()
