"""Host-side mirror of the reference's interface for the Boyer-Moore path, over the C ABI.

The reference has one program, BoyreMoore/BoyreMoore/BoyreMoore.cpp, whose stages map to:

    build_tables(pattern)              BoyreMoore.cpp:153-190   (badSymTab / goodSymTab)
    partition_words(text, P)           BoyreMoore.cpp:94-141    (start_endi)
    search_partitions(text, pattern,   x64/Debug/kernel1.cl:1   (the kernel entry `search`:
        se, gs, bs)                                              text, pattern, se, ans, gstable,
                                                                 bstable, sublength)
    search(text, pattern)              BoyreMoore.cpp:192-313   (buffers, launch, read-back) with
                                                                 ONE partition {0, n-1}: the serial
                                                                 result the north star pins parity on
    search_device(text_cuda, pattern)  BoyreMoore.cpp:258-286   (launch + count read-back only)

Everything here is a thin ctypes call into libbmx.so; there is no Python or PyTorch compute
path and no fallback.  PyTorch appears only as the owner of device memory and streams.
"""
from __future__ import annotations

import ctypes
from ctypes import c_int32, c_int64, c_uint64, c_void_p

import numpy as np

from . import _lib
from ._lib import BmxStats, check

_VARIANTS = {"auto": 0, "qgram": 1, "window": 2, "shiftand": 3}


def _variant(v, ignore_case: bool = False) -> int:
    flag = _lib.IGNORE_CASE if ignore_case else 0
    if isinstance(v, str):
        return _VARIANTS[v] | flag
    return int(v) | flag


def _as_bytes(pattern) -> bytes:
    if isinstance(pattern, str):
        return pattern.encode("latin-1")
    return bytes(pattern)


def version() -> int:
    return _lib.load().bmx_version()


def device_count() -> int:
    return _lib.load().bmx_device_count()


def build_tables(pattern) -> tuple[np.ndarray, np.ndarray]:
    """(bad[256], good[m]) for `pattern` -- BoyreMoore.cpp:153-190."""
    lib = _lib.load()
    pat = _as_bytes(pattern)
    m = len(pat)
    bad = np.zeros(256, dtype=np.int32)
    good = np.zeros(max(m, 1), dtype=np.int32)
    check(lib.bmx_build_tables(pat, m, bad.ctypes.data_as(ctypes.POINTER(c_int32)),
                               good.ctypes.data_as(ctypes.POINTER(c_int32))))
    return bad, good[:m]


def partition_words(text, nparts: int) -> np.ndarray:
    """The reference's word partitioner -- BoyreMoore.cpp:94-141.  Returns se[2*nparts]."""
    lib = _lib.load()
    buf = np.frombuffer(_as_bytes(text), dtype=np.uint8)
    se = np.zeros(2 * max(nparts, 0), dtype=np.int32)
    check(lib.bmx_partition_words(buf.ctypes.data if buf.size else None, buf.size, nparts,
                                  se.ctypes.data_as(ctypes.POINTER(c_int32))))
    return se


def _host_text(text):
    """(pointer, n, keepalive) for bytes / numpy uint8 / CPU torch uint8 tensors."""
    if isinstance(text, (bytes, bytearray, memoryview, str)):
        arr = np.frombuffer(_as_bytes(text), dtype=np.uint8)
        return (arr.ctypes.data if arr.size else None), arr.size, arr
    if isinstance(text, np.ndarray):
        arr = np.ascontiguousarray(text.view(np.uint8).reshape(-1))
        return (arr.ctypes.data if arr.size else None), arr.size, arr
    # torch CPU tensor (possibly pinned)
    t = text.contiguous().view(-1)
    if t.is_cuda:
        raise TypeError("search() takes host memory; use search_device() for CUDA tensors")
    return (t.data_ptr() if t.numel() else None), t.numel(), t


def search(text, pattern, max_positions: int | None = None, variant="auto", device: int | None = None,
           return_stats: bool = False, ignore_case: bool = False):
    """Serial-reference result for host text: (count, positions[int64]) -- BoyreMoore.cpp:192-313.

    positions holds min(count, max_positions) ascending start offsets (default: room for all).
    max_positions=0 is count-only.  ignore_case=True matches ASCII letters in either case (BMX_IGNORE_CASE):
    the result for text.lower() and pattern.lower(), without touching the text.
    """
    lib = _lib.load()
    pat = _as_bytes(pattern)
    ptr, n, keep = _host_text(text)
    if device is None:
        import torch
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    count = c_uint64(0)
    stats = BmxStats()
    # "room for all" does not mean 8 bytes per text byte: start with one hit per 64 bytes and, for the rare text
    # that is denser, fetch again with room for the count the first call reported
    open_ended = max_positions is None
    cap = _first_cap(n, len(pat)) if open_ended else int(max_positions)
    while True:
        pos = np.empty(cap, dtype=np.int64)
        check(lib.bmx_search_ex(device, ptr, n, pat, len(pat), pos.ctypes.data if cap else None,
                                cap, ctypes.byref(count), _variant(variant, ignore_case), ctypes.byref(stats)))
        if not open_ended or count.value <= cap:
            break
        cap = int(count.value)
    del keep
    out = pos[: min(count.value, cap)]
    return (count.value, out, stats.as_dict()) if return_stats else (count.value, out)


def _first_cap(n: int, m: int) -> int:
    return max(0, min(n - m + 1, max(1 << 20, n // 64)))


def search_device(text, pattern, pos_out=None, max_positions: int | None = None, pos_base: int = 0,
                  variant="auto", stream=None, timing: bool = True, ignore_case: bool = False):
    """Scan a CUDA uint8 tensor -- BoyreMoore.cpp:258-286.  Returns (count, positions, stats).

    pos_out: optional preallocated int64 CUDA tensor; otherwise max_positions (default 0 =
    count-only) entries are allocated.  positions is the filled prefix of that tensor (or None).
    Every reported position has pos_base added (multi-GPU shards report global offsets).
    timing=False skips the library's CUDA-event instrumentation (a few microseconds per call): stats is then {}.
    ignore_case=True: ASCII case-insensitive, as search(); the tensor is left as it was.
    """
    import torch

    lib = _lib.load()
    pat = _as_bytes(pattern)
    if not text.is_cuda or text.dtype != torch.uint8 or not text.is_contiguous():
        raise TypeError("search_device() needs a contiguous CUDA uint8 tensor")
    n = text.numel()
    with torch.cuda.device(text.device):
        if pos_out is None and max_positions:
            pos_out = torch.empty(int(max_positions), dtype=torch.int64, device=text.device)
        cap = 0 if pos_out is None else pos_out.numel()
        if pos_out is not None and (pos_out.dtype != torch.int64 or not pos_out.is_cuda or not pos_out.is_contiguous()):
            raise TypeError("pos_out must be a contiguous CUDA int64 tensor")
        s = stream if stream is not None else torch.cuda.current_stream(text.device)
        count = c_uint64(0)
        stats = BmxStats()
        check(lib.bmx_search_device_ex(c_void_p(text.data_ptr() if n else 0), n, pat, len(pat), c_int64(pos_base),
                                       c_void_p(pos_out.data_ptr()) if cap else None, cap, ctypes.byref(count),
                                       _variant(variant, ignore_case), ctypes.byref(stats) if timing else None,
                                       c_void_p(s.cuda_stream)))
    found = None if pos_out is None else pos_out[: min(count.value, cap)]
    return count.value, found, (stats.as_dict() if timing else {})


def search_multi(text, patterns, max_positions: int | None = None, device: int | None = None):
    """K patterns over one HOST text with a single host->device copy (SURVEY 8f: multi-pattern batching).
    Returns [(count, positions[int64])] in pattern order, each equal to search(text, pattern)."""
    lib = _lib.load()
    pats = [_as_bytes(p) for p in patterns]
    ptr, n, keep = _host_text(text)
    k = len(pats)
    caps = [_first_cap(n, len(p)) if max_positions is None else int(max_positions) for p in pats]
    c_pats = (ctypes.c_char_p * k)(*pats)
    c_ms = (c_int32 * k)(*[len(p) for p in pats])
    counts = (c_uint64 * k)()
    if device is None:
        import torch
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    while True:
        bufs = [np.empty(cap, dtype=np.int64) for cap in caps]
        c_pos = (c_void_p * k)(*[b.ctypes.data if b.size else None for b in bufs])
        c_caps = (c_int64 * k)(*caps)
        check(lib.bmx_search_multi(device, ptr, n, k, c_pats, c_ms, c_pos, c_caps, counts))
        if max_positions is not None or all(int(counts[i]) <= caps[i] for i in range(k)):
            break
        caps = [max(caps[i], int(counts[i])) for i in range(k)]      # a pattern denser than one hit per 64 bytes
    del keep
    return [(int(counts[i]), bufs[i][: min(int(counts[i]), caps[i])]) for i in range(k)]


def search_multi_device(text, patterns, max_positions: int = 0, stream=None):
    """K patterns in one pass over a CUDA uint8 tensor (bmx_search_multi_device).  Returns
    [(count, positions CUDA tensor or None)] in pattern order; max_positions entries of room per pattern (0: counts only)."""
    import torch

    lib = _lib.load()
    pats = [_as_bytes(p) for p in patterns]
    if not text.is_cuda or text.dtype != torch.uint8 or not text.is_contiguous():
        raise TypeError("search_multi_device() needs a contiguous CUDA uint8 tensor")
    k, n = len(pats), text.numel()
    with torch.cuda.device(text.device):
        outs = [torch.empty(int(max_positions), dtype=torch.int64, device=text.device) if max_positions else None for _ in pats]
        c_pats = (ctypes.c_char_p * k)(*pats)
        c_ms = (c_int32 * k)(*[len(p) for p in pats])
        c_pos = (c_void_p * k)(*[o.data_ptr() if o is not None else None for o in outs])
        c_caps = (c_int64 * k)(*[int(max_positions)] * k)
        counts = (c_uint64 * k)()
        s = stream if stream is not None else torch.cuda.current_stream(text.device)
        check(lib.bmx_search_multi_device(c_void_p(text.data_ptr() if n else 0), n, k, c_pats, c_ms, c_pos, c_caps, counts,
                                          c_void_p(s.cuda_stream)))
    return [(int(counts[i]), None if outs[i] is None else outs[i][: min(int(counts[i]), int(max_positions))]) for i in range(k)]


def find_first(text, pattern) -> int:
    """Smallest start position of pattern in HOST text, or -1 -- the early-exit "first occurrence" query of
    the vendored CUDA sample (CUDA/Parallel-Programs-master/cuda/boyer-moore/boyer-moore.cu:62-86), equal to
    search()'s first position.  Copies and scans stop after the first chunk that holds a match."""
    lib = _lib.load()
    pat = _as_bytes(pattern)
    ptr, n, keep = _host_text(text)
    first = c_int64(-1)
    check(lib.bmx_find_first(ptr, n, pat, len(pat), ctypes.byref(first)))
    del keep
    return first.value


def find_first_device(text, pattern, stream=None) -> int:
    """find_first() for a contiguous CUDA uint8 tensor (growing chunks, at most one chunk scanned in vain)."""
    import torch

    lib = _lib.load()
    pat = _as_bytes(pattern)
    if not text.is_cuda or text.dtype != torch.uint8 or not text.is_contiguous():
        raise TypeError("find_first_device() needs a contiguous CUDA uint8 tensor")
    n = text.numel()
    first = c_int64(-1)
    with torch.cuda.device(text.device):
        s = stream if stream is not None else torch.cuda.current_stream(text.device)
        check(lib.bmx_find_first_device(c_void_p(text.data_ptr() if n else 0), n, pat, len(pat), ctypes.byref(first),
                                        c_void_p(s.cuda_stream)))
    return first.value


def search_partitions(text, pattern, se, gs=None, bs=None) -> np.ndarray:
    """Mirror of the kernel entry `search` (kernel1.cl:1): per-range counts ans[nparts]."""
    lib = _lib.load()
    pat = _as_bytes(pattern)
    ptr, n, keep = _host_text(text)
    se = np.ascontiguousarray(se, dtype=np.int32)
    nparts = se.size // 2
    if nparts and int(se[1::2].max()) >= n:
        raise ValueError("a partition ends beyond the text")
    ans = np.zeros(nparts, dtype=np.int32)
    p32 = ctypes.POINTER(c_int32)
    gs_a = None if gs is None else np.ascontiguousarray(gs, dtype=np.int32)
    bs_a = None if bs is None else np.ascontiguousarray(bs, dtype=np.int32)
    check(lib.bmx_search_partitions(ptr, pat, se.ctypes.data_as(p32), ans.ctypes.data_as(p32),
                                    None if gs_a is None else gs_a.ctypes.data_as(p32),
                                    None if bs_a is None else bs_a.ctypes.data_as(p32), len(pat), nparts))
    del keep
    return ans


def search_ranges(text, pattern, begin, end, max_positions: int | None = None, device: int | None = None):
    """Many ranges of one HOST text in one pass (bmx_search_ranges) -- the kernel entry `search` (kernel1.cl:1)
    for any number of half-open ranges [begin[d], end[d]), with positions.  Returns (counts, offsets, positions):

        counts[d]     matches lying fully inside range d (= search(text[begin[d]:end[d]], pattern)[0])
        offsets       nranges + 1 entries, offsets[d] = counts[:d].sum(), offsets[-1] = total
        positions     range d's starts, RELATIVE TO begin[d], at positions[offsets[d]:offsets[d+1]] (the first
                      min(total, max_positions) entries of that concatenation)

    max_positions=None: room for all (grown like search()); 0: counts only (positions is empty).
    A ragged batch held as values + offsets o is one call:

        counts, offs, pos = search_ranges(values, pattern, begin=o[:-1], end=o[1:])
    """
    lib = _lib.load()
    pat = _as_bytes(pattern)
    ptr, n, keep = _host_text(text)
    b = np.ascontiguousarray(begin, dtype=np.int64).reshape(-1)
    e = np.ascontiguousarray(end, dtype=np.int64).reshape(-1)
    if b.size != e.size:
        raise ValueError("begin and end must have the same length")
    if device is None:
        import torch
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    d = b.size
    counts = np.zeros(d, dtype=np.uint64)
    offsets = np.zeros(d + 1, dtype=np.int64)
    open_ended = max_positions is None
    cap = _first_cap(n, len(pat)) if open_ended else int(max_positions)
    while True:
        pos = np.empty(cap, dtype=np.int64)
        check(lib.bmx_search_ranges(device, ptr, n, d, b.ctypes.data if d else None, e.ctypes.data if d else None, pat, len(pat),
                                    pos.ctypes.data if cap else None, cap, counts.ctypes.data if d else None, offsets.ctypes.data))
        total = int(offsets[-1])
        if not open_ended or total <= cap:
            break
        cap = total
    del keep
    return counts, offsets, pos[: min(total, cap)]


def search_ranges_device(text, pattern, begin, end, max_positions: int = 0, stream=None):
    """search_ranges() for CUDA tensors (bmx_search_ranges_device): a contiguous uint8 text and int64 begin / end on
    the same device.  Returns (counts int64, offsets int64 [nranges + 1], positions or None) as CUDA tensors;
    positions is the filled prefix of a tensor of max_positions entries (0 = counts only).  Ragged batch:

        counts, offs, pos = search_ranges_device(values, pattern, offs_in[:-1], offs_in[1:], max_positions=k)

    A range outside [0, len(text)] raises BmxError (BMX_E_BADARG); the library stays usable.
    """
    import torch

    lib = _lib.load()
    pat = _as_bytes(pattern)
    if not text.is_cuda or text.dtype != torch.uint8 or not text.is_contiguous():
        raise TypeError("search_ranges_device() needs a contiguous CUDA uint8 tensor")
    for t in (begin, end):
        if not t.is_cuda or t.dtype != torch.int64 or t.dim() != 1 or t.device != text.device:
            raise TypeError("begin / end must be 1-D CUDA int64 tensors on the text's device")
    if begin.numel() != end.numel():
        raise ValueError("begin and end must have the same length")
    begin, end = begin.contiguous(), end.contiguous()
    n, d, cap = text.numel(), begin.numel(), int(max_positions)
    with torch.cuda.device(text.device):
        counts = torch.empty(d, dtype=torch.int64, device=text.device)
        offsets = torch.empty(d + 1, dtype=torch.int64, device=text.device)
        pos = torch.empty(cap, dtype=torch.int64, device=text.device) if cap else None
        s = stream if stream is not None else torch.cuda.current_stream(text.device)
        total = c_uint64(0)
        check(lib.bmx_search_ranges_device(c_void_p(text.data_ptr() if n else 0), n, d, c_void_p(begin.data_ptr() if d else 0),
                                           c_void_p(end.data_ptr() if d else 0), pat, len(pat),
                                           c_void_p(pos.data_ptr()) if cap else None, cap,
                                           c_void_p(counts.data_ptr() if d else 0), c_void_p(offsets.data_ptr()),
                                           ctypes.byref(total), c_void_p(s.cuda_stream)))
    return counts, offsets, None if pos is None else pos[: min(total.value, cap)]


def _check_cuda(t, dtype: str, what: str):
    """The scanner takes raw device pointers: a CPU, strided or wrongly typed tensor would be read as other bytes."""
    import torch

    if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != getattr(torch, dtype) or not t.is_contiguous():
        raise TypeError(f"{what} must be a contiguous CUDA {dtype} tensor")


class Scanner:
    """Reusable scanner (bmx_scanner_*): pattern block + look-back scratch kept across scans."""

    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        self._h = c_void_p()
        check(self._lib.bmx_scanner_create(device, ctypes.byref(self._h)))

    def close(self):
        if self._h:
            self._lib.bmx_scanner_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_pattern(self, pattern, variant="auto", stream=0, ignore_case: bool = False):
        """ignore_case=True: the following scans match ASCII letters in either case (BMX_IGNORE_CASE)."""
        pat = _as_bytes(pattern)
        check(self._lib.bmx_scanner_set_pattern(self._h, pat, len(pat), _variant(variant, ignore_case), c_void_p(stream)))

    def begin(self, pos_out=None, stream=0):
        if pos_out is not None:
            _check_cuda(pos_out, "int64", "Scanner.begin(): pos_out")
        cap = 0 if pos_out is None else pos_out.numel()
        check(self._lib.bmx_scanner_begin(self._h, c_void_p(pos_out.data_ptr()) if cap else None, cap, c_void_p(stream)))

    def scan(self, text, pos_base=0, stream=0):
        _check_cuda(text, "uint8", "Scanner.scan(): text")
        check(self._lib.bmx_scanner_scan(self._h, c_void_p(text.data_ptr()), text.numel(), c_int64(pos_base), c_void_p(stream)))

    def set_timing(self, level: int):
        """0: no CUDA events, 1: whole scan (device_ms), 2: also the scan kernel alone (default)."""
        check(self._lib.bmx_scanner_set_timing(self._h, int(level)))

    def export_result(self, packed, stream=0):
        """Enqueue {count, positions written, first len(packed)-2 positions} into the int64 CUDA
        tensor `packed` (no host sync): the send buffer of the multi-GPU exchange step."""
        _check_cuda(packed, "int64", "Scanner.export_result(): packed")
        check(self._lib.bmx_scanner_export_result(self._h, c_void_p(packed.data_ptr()), packed.numel() - 2, c_void_p(stream)))

    def finish(self, stream=0):
        count = c_uint64(0)
        stats = BmxStats()
        check(self._lib.bmx_scanner_finish(self._h, ctypes.byref(count), ctypes.byref(stats), c_void_p(stream)))
        return count.value, stats.as_dict()


class Dictionary:
    """A compiled pattern set for dictionary search (bmx_dict_*; `grep -F -f wordlist`): 1 .. 65536 patterns of
    7 .. 4096 bytes each, hashed and uploaded once to `device`, then searched in one pass per text.

    A match is a pair (p, k) with text[p:p+len(patterns[k])] == patterns[k]; the pairs come sorted by p, then k
    (duplicate patterns are each reported).  counts[k] is exact and equals search(text, patterns[k])[0].  The
    handle is immutable: several threads may search with it at once, each on its own stream.
    """

    def __init__(self, patterns, device: int = 0):
        self._lib = _lib.load()
        self._h = c_void_p()
        pats = [_as_bytes(p) for p in patterns]
        self.npat, self.device = len(pats), int(device)
        self.min_length = min((len(p) for p in pats), default=0)
        c_pats = (ctypes.c_char_p * self.npat)(*pats)
        c_ms = (c_int32 * self.npat)(*[len(p) for p in pats])
        check(self._lib.bmx_dict_create(self.device, self.npat, c_pats, c_ms, ctypes.byref(self._h)))

    def close(self):
        if self._h:
            self._lib.bmx_dict_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def search(self, text, max_matches: int | None = None):
        """HOST text (copied to the device once) -> (counts uint64[K], positions int64, pattern_ids int32, total).
        positions / pattern_ids hold the first min(total, max_matches) pairs; None: room for all; 0: counts only."""
        ptr, n, keep = _host_text(text)
        counts = np.zeros(self.npat, dtype=np.uint64)
        total = c_uint64(0)
        open_ended = max_matches is None
        cap = _first_cap(n, self.min_length) if open_ended else int(max_matches)
        while True:
            pos = np.empty(cap, dtype=np.int64)
            pat = np.empty(cap, dtype=np.int32)
            check(self._lib.bmx_dict_search(self._h, ptr, n, pos.ctypes.data if cap else None, pat.ctypes.data if cap else None,
                                            cap, counts.ctypes.data, ctypes.byref(total)))
            if not open_ended or total.value <= cap:
                break
            cap = int(total.value)
        del keep
        k = min(total.value, cap)
        return counts, pos[:k], pat[:k], total.value

    def search_device(self, text, max_matches: int = 0, pos_base: int = 0, stream=None):
        """A contiguous CUDA uint8 tensor on the dictionary's device -> (counts uint64[K] on the host, positions int64
        and pattern_ids int32 CUDA tensors holding the first min(total, max_matches) pairs or None, total).
        Every position has pos_base added; max_matches=0 is counts only."""
        import torch

        _check_cuda(text, "uint8", "Dictionary.search_device(): text")
        n, cap = text.numel(), int(max_matches)
        counts = np.zeros(self.npat, dtype=np.uint64)
        total = c_uint64(0)
        with torch.cuda.device(text.device):
            pos = torch.empty(cap, dtype=torch.int64, device=text.device) if cap else None
            pat = torch.empty(cap, dtype=torch.int32, device=text.device) if cap else None
            s = stream if stream is not None else torch.cuda.current_stream(text.device)
            check(self._lib.bmx_dict_search_device(self._h, c_void_p(text.data_ptr() if n else 0), n, c_int64(pos_base),
                                                   c_void_p(pos.data_ptr()) if cap else None, c_void_p(pat.data_ptr()) if cap else None,
                                                   cap, counts.ctypes.data, ctypes.byref(total), c_void_p(s.cuda_stream)))
        k = min(total.value, cap)
        return counts, None if pos is None else pos[:k], None if pat is None else pat[:k], total.value


class Exchange:
    """The exchange step of the sharded scan over NVLink peer memory (bmx_exchange_*): one per rank (= GPU).

    post(scanner) ships the scanner's running result {count, list} as the next step, collect() completes the
    oldest uncollected step (rank dst also concatenates the lists into `out`), wait(seq) blocks the host until
    that step has been collected here and returns (total, per-rank counts, gathered length).  post/collect only
    enqueue a kernel; nothing synchronises with the host except wait().
    """

    HANDLE_BYTES = 64

    def __init__(self, device: int, rank: int, world: int, dst: int = 0, head_cap: int = 4096, tail_cap: int = 0, depth: int = 4):
        self._lib = _lib.load()
        self._h = c_void_p()
        self.rank, self.world, self.dst = rank, world, dst
        check(self._lib.bmx_exchange_create(device, rank, world, dst, head_cap, tail_cap, depth, ctypes.byref(self._h)))

    def close(self):
        if self._h:
            self._lib.bmx_exchange_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def handle(self) -> bytes:
        buf = ctypes.create_string_buffer(self.HANDLE_BYTES)
        check(self._lib.bmx_exchange_handle(self._h, buf))
        return buf.raw

    def connect(self, handles: bytes):
        """handles: world x 64 bytes in rank order (this rank's own entry is ignored)."""
        assert len(handles) == self.world * self.HANDLE_BYTES
        check(self._lib.bmx_exchange_connect(self._h, handles))

    @staticmethod
    def connect_local(exchanges):
        """All ranks live in this process: wire them up directly (peer access is enabled as needed)."""
        arr = (c_void_p * len(exchanges))(*[x._h for x in exchanges])
        check(_lib.load().bmx_exchange_connect_local(arr, len(exchanges)))

    def post(self, scanner, stream=0) -> int:
        seq = c_uint64(0)
        check(self._lib.bmx_exchange_post(self._h, scanner._h, c_void_p(stream), ctypes.byref(seq)))
        return seq.value

    def collect(self, out=None, stream=0) -> int:
        seq = c_uint64(0)
        cap = 0 if out is None else out.numel()
        check(self._lib.bmx_exchange_collect(self._h, c_void_p(out.data_ptr()) if cap else None, cap, c_void_p(stream), ctypes.byref(seq)))
        return seq.value

    def wait(self, seq: int):
        total, gathered = c_uint64(0), c_int64(0)
        counts = (c_uint64 * self.world)()
        check(self._lib.bmx_exchange_wait(self._h, seq, ctypes.byref(total), counts, ctypes.byref(gathered)))
        return total.value, [int(c) for c in counts], gathered.value


class MultiGpu:
    """Single-process multi-GPU search over host text (bmx_mg_*): shards + (m-1) halo, one host thread per GPU."""

    def __init__(self, ngpus: int = 0):
        self._lib = _lib.load()
        self._h = c_void_p()
        check(self._lib.bmx_mg_create(ngpus, ctypes.byref(self._h)))
        self.ngpus = self._lib.bmx_mg_device_count(self._h)

    def close(self):
        if self._h:
            self._lib.bmx_mg_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def search(self, text, pattern, max_positions: int | None = None):
        """(count, positions, per_gpu_counts) -- the serial-reference result, like search()."""
        pat = _as_bytes(pattern)
        ptr, n, keep = _host_text(text)
        open_ended = max_positions is None
        cap = _first_cap(n, len(pat)) if open_ended else int(max_positions)
        count = c_uint64(0)
        shard = (c_uint64 * self.ngpus)()
        while True:
            pos = np.empty(cap, dtype=np.int64)
            check(self._lib.bmx_mg_search(self._h, ptr, n, pat, len(pat), pos.ctypes.data if cap else None,
                                          cap, ctypes.byref(count), shard))
            if not open_ended or count.value <= cap:
                break
            cap = int(count.value)
        del keep
        return count.value, pos[: min(count.value, cap)], [int(x) for x in shard]

    def search_device(self, shards, pos_bases, pattern, pos_out=None):
        """Device-resident shards (CUDA uint8 tensors, shard r on GPU r, own range + (m-1)-byte halo) ->
        (count, positions on GPU 0 or None, per_gpu_counts); the exchange step runs inside the library over
        peer memory (bmx_mg_search_device)."""
        pat = _as_bytes(pattern)
        assert len(shards) == self.ngpus == len(pos_bases)
        ptrs = (c_void_p * self.ngpus)(*[t.data_ptr() if t.numel() else None for t in shards])
        ns = (c_int64 * self.ngpus)(*[t.numel() for t in shards])
        bases = (c_int64 * self.ngpus)(*[int(b) for b in pos_bases])
        cap = 0 if pos_out is None else pos_out.numel()
        count = c_uint64(0)
        shard = (c_uint64 * self.ngpus)()
        check(self._lib.bmx_mg_search_device(self._h, ptrs, ns, bases, pat, len(pat), c_void_p(pos_out.data_ptr()) if cap else None,
                                             cap, ctypes.byref(count), shard))
        found = None if pos_out is None else pos_out[: min(count.value, cap)]
        return count.value, found, [int(x) for x in shard]
