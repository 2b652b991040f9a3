"""The exchange step of the sharded scan with a different result in every step.

The exchange keeps state from step to step: a header/head ring of `depth` slots (slot = seq % depth), two tail areas
per source on dst (seq % 2), a host-mapped result ring of `depth` entries, and the count word of each posted scanner
(the carry slot of its last scan, the count-only running total, or the zero word when nothing was scanned).  When
every step carries the same result, a collect that reads another step's slot or tail area, or a wait that reads
another step's result entry, still returns the right answer.  Here every step has its own text and pattern, every
rank its own density, shard shape, chain of scans and output buffer, and the generator asserts before anything runs
that rank r's (count, list) in step q differs from its values in steps q-1, q-2 (same tail area) and q-depth (same
head slot and result entry).  KMP on the whole text of the step is the truth.

The list on dst follows one rule in both exchanges, the library's (bmx_exchange_*) and combine_hits over
torch.distributed: rank r ships s_r = min(count_r, held_r, room) entries, where held_r is what its own buffer holds
and room is head_cap + tail_cap (unbounded for combine_hits), and the list stops behind the first rank with
s_r != count_r.  That makes it a prefix of the global ascending list."""
from __future__ import annotations

import os
import socket
import sys
from ctypes import byref, c_int64, c_uint64, c_void_p
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

torch = pytest.importorskip("torch")

from test_emission_contract_gpu import G, assert_same, expect, guarded, lib_of, ok  # noqa: E402
from test_exact_reference import kmp  # noqa: E402

TAIL_AREAS = 2                                  # kTailDepth in bmx_exchange.cu
BG = np.frombuffer(b"bcd", dtype=np.uint8)      # background bytes: no 'a', so every hit of 'a' * m is planted


def shipped(counts, held, room):
    """Entries of each rank's list in the gathered list: s_r = min(count_r, held_r, room) for every rank up to and
    including the first one with s_r != count_r, 0 behind it."""
    take, complete = [], True
    for c, h in zip(counts, held):
        s = min(c, h, room)
        take.append(s if complete else 0)
        complete = complete and s == c
    return take


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


# ---------------------------------------------------------------------------------------------------------------
# Step generator (CPU): one text and pattern per step, one shard shape, density, chain and position buffer per rank
# ---------------------------------------------------------------------------------------------------------------
class Step:
    """Rank r owns the starts [cut[r], cut[r+1]) and scans text[cut[r]:cut[r+1] + m - 1] (an 'empty' rank scans 0 bytes)
    as a chain of pieces; pos_cap[r] is None (count-only), 0 (a pointer with no room) or the size of its buffer."""

    def __init__(self, text, pat, cut, shape, kind, pieces, pos_cap, truth):
        self.text, self.pat, self.cut, self.shape, self.kind = text, pat, cut, shape, kind
        self.pieces, self.pos_cap, self.truth = pieces, pos_cap, truth
        self.m = len(pat)
        ends = np.searchsorted(truth, cut)
        self.lists = [truth[ends[r]:ends[r + 1]] for r in range(len(cut) - 1)]
        self.counts = [int(x.size) for x in self.lists]
        self.held = [0 if c is None else min(n, c) for n, c in zip(self.counts, pos_cap)]

    def read_range(self, r):
        if self.shape[r] == "empty":
            return self.cut[r], self.cut[r]
        return self.cut[r], min(self.text.size, self.cut[r + 1] + self.m - 1)

    def expected(self, room):
        take = shipped(self.counts, self.held, room)
        return self.truth[:sum(take)]


def make_step(oracle, rng, world, no_zero, dense_ok):
    """A random step.  no_zero[r]: rank r must have hits (it had none in a step it is compared with)."""
    m = int(rng.choice([1, 2, 3, 4, 5, 7, 8, 12, 16]))
    shape, kind, lens = [], [], []
    for r in range(world):
        sh = "normal" if no_zero[r] or world == 1 else str(rng.choice(["normal"] * 6 + ["empty", "short"]))
        kinds = ["few", "seams"] + (["dense"] if dense_ok else []) + ([] if no_zero[r] else ["none"])
        k = str(rng.choice(kinds)) if sh == "normal" else "none"
        shape.append(sh)
        kind.append(k)
        lens.append(0 if sh != "normal" else int(rng.integers(4200, 9000)) if k == "dense" else int(rng.integers(300, 3000)) | 1)
    cut = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    n = int(cut[-1]) + m - 1
    text = rng.choice(BG, size=n)
    for r in range(world):
        lo, hi = int(cut[r]), int(cut[r + 1])
        if kind[r] == "few":
            starts = rng.integers(lo, hi, size=int(rng.integers(1, 13)))
        elif kind[r] == "seams":          # the first and last own start, a run ending on the seam, one inside
            starts = [lo, hi - 1, max(lo, hi - m), int(rng.integers(lo, hi))]
        elif kind[r] == "dense":          # a one-byte run: thousands of hits, past any head_cap here
            d = int(rng.integers(4100, hi - lo))
            a = int(rng.integers(lo, hi - d + 1))
            text[a:a + d + m - 1] = ord("a")
            starts = []
        else:
            starts = []
        for s in starts:
            text[s:s + m] = ord("a")
    pieces, pos_cap = [], []
    truth = kmp(oracle, text, b"a" * m)
    for r in range(world):
        lo, hi = int(cut[r]), int(cut[r + 1])
        k = int(rng.integers(1, 4)) if hi - lo >= 64 else 1
        inner = sorted({lo + (int(x) | 1) for x in rng.integers(1, hi - lo - 2, size=k - 1)}) if k > 1 else []
        pieces.append([lo] + inner + [hi])
        c = int(((truth >= lo) & (truth < hi)).sum())
        pick = rng.random()
        if pick < 0.12:
            pos_cap.append(None)
        elif pick < 0.2:
            pos_cap.append(0)
        elif pick < 0.35 and c > 1:
            pos_cap.append(int(rng.integers(1, c)))
        else:
            pos_cap.append(c + int(rng.integers(0, 40)))
    return Step(text, b"a" * m, cut, shape, kind, pieces, pos_cap, truth)


def _key(step, r):
    return step.counts[r], step.lists[r].tobytes()


def make_steps(oracle, seed, world, depth, n_steps, dense_ok=True):
    """n_steps steps (index 0 = seq 1) in which every rank's (count, list) differs from its own in the steps that share
    a tail area (q-2), a head slot and a result entry (q-depth), and from the step before (q-1)."""
    rng = np.random.default_rng(seed)
    steps = []
    for q in range(n_steps):
        lags = [q - d for d in {1, TAIL_AREAS, depth} if q - d >= 0]
        no_zero = [any(steps[j].counts[r] == 0 for j in lags) for r in range(world)]
        for _attempt in range(50):
            st = make_step(oracle, rng, world, no_zero, dense_ok)
            if all(_key(st, r) != _key(steps[j], r) for j in lags for r in range(world)):
                break
        for j in lags:                  # the shape of the test, asserted on the truth before anything runs
            for r in range(world):
                assert _key(st, r) != _key(steps[j], r), (q, j, r)
        steps.append(st)
    return steps


def test_step_generator_distinct_and_covering(oracle):
    """CPU: the generated steps satisfy the distinctness rule and reach what the GPU tests rely on: empty and (m-1)-byte
    shards, every density, chains of 1, 2 and 3 scans with hits in the last piece, count-only ranks and ranks capped
    below their count in the same step as ranks that ship lists, and dense ranks past 4096 hits."""
    steps = make_steps(oracle, 7, 5, 3, 40)
    seen = set()
    for st in steps:
        assert sum(st.counts) == st.truth.size
        for r in range(5):
            seen.add(st.shape[r])
            seen.add(st.kind[r])
            seen.add(("pieces", len(st.pieces[r]) - 1))
            lo, hi = st.pieces[r][-2], st.pieces[r][-1]
            if len(st.pieces[r]) == 3 and ((st.truth >= lo) & (st.truth < hi)).any() and st.pos_cap[r] is not None:
                seen.add("chain-2-hits-in-last-piece")
            if st.kind[r] == "dense" and st.counts[r] > 4096:
                seen.add("dense>4096")
        caps = st.pos_cap
        if None in caps and any(c is not None and c >= n > 0 for c, n in zip(caps, st.counts)):
            seen.add("count-only-next-to-list")
        if any(c is not None and c < n for c, n in zip(caps, st.counts)):
            seen.add("capped")
    want = {"normal", "empty", "short", "none", "few", "seams", "dense", ("pieces", 1), ("pieces", 2), ("pieces", 3),
            "chain-2-hits-in-last-piece", "dense>4096", "count-only-next-to-list", "capped"}
    assert want <= seen, want - seen


def test_prefix_rule_is_the_uniform_one(bmx, oracle):
    """CPU: with one cap for every rank, shipped() gives the prefix test_exchange_gpu._expected_prefix gives."""
    from parallel_implementation_of_string_matching_algorithms_opencl_b200 import distributed as bd
    from test_exchange_gpu import _expected_prefix, _make_text
    for world, head, tail, local in ((2, 4096, 0, 1 << 16), (4, 4, 16, 1 << 12), (3, 16, 1 << 12, 20), (3, 64, 0, 0)):
        text, pat = _make_text(bmx, 50_003, 9, 5 + world, "dna", 60, world)
        want, counts, prefix = _expected_prefix(oracle, text, pat, world, head, tail, local, 1 << 30)
        ranges = [bd.shard_bounds(text.size, world, r) for r in range(world)]
        assert counts == [int(((want >= lo) & (want < hi)).sum()) for lo, hi in ranges]
        assert sum(shipped(counts, [min(c, local) for c in counts], head + tail)) == prefix.size


# ---------------------------------------------------------------------------------------------------------------
# 1. The library exchange, all ranks in this process (round-robin over the visible GPUs, one stream each)
# ---------------------------------------------------------------------------------------------------------------
class World:
    def __init__(self, bmx, world, dst, depth, head_cap, tail_cap, steps):
        self.bmx, self.lib = bmx, lib_of(bmx)
        self.world, self.dst, self.depth = world, dst, depth
        self.room, self.tail_cap = head_cap + tail_cap, tail_cap
        self.steps = steps
        ngpu = torch.cuda.device_count()
        self.devices = [r % ngpu for r in range(world)]
        self.streams, self.scanners, self.xs = [], [], []
        for r in range(world):
            with torch.cuda.device(self.devices[r]):
                self.streams.append(torch.cuda.Stream(device=self.devices[r]))
                self.scanners.append(bmx.Scanner(self.devices[r]))
                self.xs.append(bmx.Exchange(self.devices[r], r, world, dst=dst, head_cap=head_cap, tail_cap=tail_cap,
                                            depth=depth))
        bmx.Exchange.connect_local(self.xs)
        self.live = {}                  # seq -> device buffers the step's kernels use, and dst's output
        self.checked = 0

    def post(self, q):
        """Scan step q (seq q) on every rank, as a chain of pieces, and post it."""
        st_q = self.steps[q - 1]
        keep, m = [], st_q.m
        for r in range(self.world):
            dev = torch.device("cuda", self.devices[r])
            s = self.streams[r]
            with torch.cuda.device(dev):
                a, b = st_q.read_range(r)
                td = torch.from_numpy(st_q.text[a:b].copy()).to(dev)
                cap = st_q.pos_cap[r]
                pos = None if cap is None else torch.empty(max(cap, 1), dtype=torch.int64, device=dev)
                s.wait_stream(torch.cuda.current_stream(dev))
                keep += [td, pos]
                sc = self.scanners[r]
                sc.set_pattern(st_q.pat, stream=s.cuda_stream)
                self.bmx._lib.check(self.lib.bmx_scanner_begin(sc._h, None if pos is None else c_void_p(pos.data_ptr()),
                                                               cap or 0, c_void_p(s.cuda_stream)))
                if st_q.shape[r] == "normal":
                    cuts = st_q.pieces[r]
                    for k in range(len(cuts) - 1):
                        lo, hi = cuts[k] - a, min(cuts[k + 1] + m - 1 - a, td.numel())
                        sc.scan(td[lo:hi], cuts[k], stream=s.cuda_stream)
                else:
                    sc.scan(td, a, stream=s.cuda_stream)   # 0 or m - 1 bytes: nothing launches, the zero word is posted
                assert self.xs[r].post(sc, s.cuda_stream) == q
        self.live[q] = [keep, None]

    def collect(self, q, cap="auto"):
        """Collect step q on every rank; dst writes into a guarded buffer (cap None: a NULL output), out[0] 16-byte
        aligned in odd steps and 8-byte aligned only in even ones."""
        st_q = self.steps[q - 1]
        offset = G + (q & 1 ^ 1)
        if cap == "auto":
            ends = np.cumsum(st_q.counts)
            k = st_q.expected(self.room).size
            options = sorted({int(c) + d for c in list(ends) + [k] for d in (-1, 0, 1) if c + d >= 0} | {0, 1})
            rng = np.random.default_rng(q)
            cap = None if rng.random() < 0.1 else int(rng.choice(options))
        dev = torch.device("cuda", self.devices[self.dst])
        out = None if cap is None else guarded(offset + cap + G, dev)
        for r in range(self.world):
            s = self.streams[r]
            with torch.cuda.device(self.devices[r]):
                s.wait_stream(torch.cuda.current_stream(self.devices[r]))
                ptr = c_void_p(out.data_ptr() + 8 * offset) if r == self.dst and out is not None else None
                seq = c_uint64()
                self.bmx._lib.check(self.lib.bmx_exchange_collect(self.xs[r]._h, ptr, cap if ptr else 0,
                                                                  c_void_p(s.cuda_stream), byref(seq)))
                assert seq.value == q
        self.live[q][1] = (out, cap, offset)

    def wait_check(self, q):
        """Wait for step q on every rank and check it: counts and total everywhere, the gathered prefix on dst, and
        the sentinel everywhere else in dst's buffer."""
        st_q = self.steps[q - 1]
        got = [self.xs[r].wait(q) for r in range(self.world)]
        for d in set(self.devices):
            torch.cuda.synchronize(d)
        out, cap, offset = self.live[q][1]
        prefix = st_q.expected(self.room)
        k = 0 if cap is None else min(prefix.size, cap)
        for r in range(self.world):
            total, counts, glen = got[r]
            assert total == st_q.truth.size and counts == st_q.counts, (q, r, total, counts, st_q.counts)
            assert glen == (k if r == self.dst else 0), (q, r, glen, k)
        if out is not None:
            buf = out.cpu().numpy()
            assert_same(buf, expect(buf.size, [(offset, prefix[:k])]), ("step", q, "cap", cap))
        del self.live[q]
        self.checked += 1

    def close(self):
        for d in set(self.devices):
            torch.cuda.synchronize(d)
        for x in self.xs:
            x.close()
        for sc in self.scanners:
            sc.close()


def run_order(w, order, n):
    if order == "lockstep":
        for q in range(1, n + 1):
            w.post(q)
            w.collect(q)
            w.wait_check(q)
    elif order == "pipelined":          # bench.py's order: post q, then collect q-1
        for q in range(1, n + 1):
            w.post(q)
            if q > 1:
                w.collect(q - 1)
                w.wait_check(q - 1)
        w.collect(n)
        w.wait_check(n)
    else:                               # burst: as many posts as the API allows, then every collect, then the waits
        burst = min(w.depth - 1, TAIL_AREAS) if w.tail_cap > 0 else w.depth - 1
        q, up = 1, True
        while q <= n:
            group = list(range(q, min(n, q + burst - 1) + 1))
            for p in group:
                w.post(p)
            for p in group:
                w.collect(p)
            for p in (group if up else group[::-1]):
                w.wait_check(p)
            q, up = group[-1] + 1, not up
    assert w.checked == n


# (world, dst, depth, head_cap, tail_cap, order, steps): together every value of each
ROWS = [
    (1, 0, 2, 7, 64, "lockstep", 8),
    (2, 1, 3, 4096, 0, "pipelined", 10),
    (3, 1, 4, 1, 1 << 17, "pipelined", 10),
    (5, 4, 64, 7, 1, "lockstep", 70),
    (5, 2, 4, 0, 1 << 17, "burst", 12),
    (16, 15, 3, 4096, 64, "pipelined", 9),
    (16, 7, 2, 7, 0, "lockstep", 8),
    (3, 0, 64, 1, 0, "burst", 130),
    (2, 0, 3, 0, 1, "burst", 9),
    (5, 0, 2, 4096, 1 << 17, "lockstep", 8),
    (3, 2, 4, 7, 1 << 17, "lockstep", 9),
    (16, 0, 4, 1, 1, "burst", 9),
    (2, 0, 64, 0, 0, "pipelined", 68),
]


@pytest.mark.gpu
@pytest.mark.parametrize("world,dst,depth,head_cap,tail_cap,order,n_steps", ROWS,
                         ids=[f"w{r[0]}-dst{r[1]}-d{r[2]}-h{r[3]}-t{r[4]}-{r[5]}" for r in ROWS])
def test_exchange_distinct_steps(bmx, oracle, world, dst, depth, head_cap, tail_cap, order, n_steps):
    """Every step its own text, pattern, shard shapes and buffers; every step checked against KMP."""
    steps = make_steps(oracle, 1000 * world + 10 * depth + dst, world, depth, n_steps)
    assert any(st.counts[r] > head_cap for st in steps for r in range(world)), "no step uses the tail area"
    w = World(bmx, world, dst, depth, head_cap, tail_cap, steps)
    try:
        run_order(w, order, n_steps)
    finally:
        w.close()


@pytest.mark.gpu
def test_exchange_host_side_edges(bmx, oracle):
    """The host checks of post, collect and wait (none of them launches a kernel), and a wait at the far edge of the
    result ring.  Every refused call leaves the exchange usable: the steps around it are checked as usual."""
    from parallel_implementation_of_string_matching_algorithms_opencl_b200._lib import BMX_E_BADARG, BmxError

    def refused(fn, *args, match=None):
        with pytest.raises(BmxError) as e:
            fn(*args)
        assert e.value.code == BMX_E_BADARG, e.value
        if match:
            assert match in str(e.value), e.value

    depth = 3
    steps = make_steps(oracle, 99, 2, depth, 12)
    w = World(bmx, 2, 1, depth, 16, 0, steps)
    try:
        for x in w.xs:
            refused(x.collect, None, 0)                     # nothing posted yet
            refused(x.wait, 0)
            refused(x.wait, 1)                              # not collected
        w.post(1)
        w.post(2)                                           # depth - 1 steps outstanding: the most allowed
        for r in range(2):
            refused(w.xs[r].post, w.scanners[r], w.streams[r].cuda_stream)
            refused(w.xs[r].wait, 1)                        # posted, not collected
        w.collect(1)
        w.collect(2)
        for x in w.xs:
            refused(x.collect, None, 0)                     # everything posted is collected
            refused(x.wait, 3)
        w.wait_check(2)
        w.wait_check(1)
        for q in range(3, 6):                               # collect up to 1 + depth + 1 ...
            w.post(q)
            w.collect(q)
        for d in set(w.devices):
            torch.cuda.synchronize(d)
        for x in w.xs:                                      # ... step 5 reused the entry of step 2; step 3 is at the edge
            refused(x.wait, 2, match="overwritten")
        w.wait_check(3)
        w.wait_check(4)
        w.wait_check(5)
        for x in w.xs:
            refused(x.wait, 1, match="overwritten")         # entry of step 1 now holds step 4
    finally:
        w.close()

    w = World(bmx, 2, 0, 4, 4, 64, steps)                   # a tail area: two outstanding steps at most, at any depth
    try:
        w.post(1)
        w.post(2)
        for r in range(2):
            refused(w.xs[r].post, w.scanners[r], w.streams[r].cuda_stream)
        w.collect(1)
        w.post(3)
        w.collect(2)
        w.collect(3)
        for q in (3, 2, 1):
            w.wait_check(q)
    finally:
        w.close()


# ---------------------------------------------------------------------------------------------------------------
# 2. bmx_mg_search_device: one MultiGpu across calls (its exchange and sequence numbers persist)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_mg_search_device_across_calls(bmx, oracle):
    """One MultiGpu for a sequence of searches: sparse, dense, sparse, no hits, dense again, each with several caps.
    The exchange keeps running through its depth-4 ring across calls; the first dense call grows the tail area and
    recreates the exchange, so the calls behind it restart the numbering.  Guarded output on GPU 0 every time."""
    from parallel_implementation_of_string_matching_algorithms_opencl_b200 import distributed as bd
    from test_exchange_gpu import _make_text

    lib = lib_of(bmx)
    mg = bmx.MultiGpu(0)
    R = mg.ngpus
    calls = []
    for i, kind in enumerate(("sparse", "dense", "sparse", "none", "dense")):
        text, pat = _make_text(bmx, 600_011 + 1000 * i, 8 + i, 30 + i, "dna", 40 + 10 * i, R)
        if kind == "dense":
            lo = 50_000 + 20_000 * i
            text[lo:lo + 9000 + 3000 * i] = ord("G")      # more than 4096 hits in one shard: the tail is needed
            pat = b"G" * (5 + i)
        elif kind == "none":
            pat = b"TTTTTTTTTTTTTTTTTTTTTTTTTTTTTTTT"
            assert kmp(oracle, text, pat).size == 0
        calls.append((kind, text, pat))
    prev = None
    for kind, text, pat in calls:
        m = len(pat)
        want = kmp(oracle, text, pat)
        assert (want.size == 0) == (kind == "none") and (kind != "dense" or want.size > 4096)
        assert prev is None or want.size != prev.size
        prev = want
        shards, bases, ends = [], [], []
        for r in range(R):
            lo, hi = bd.shard_bounds(text.size, R, r)
            ends.append(int(np.searchsorted(want, hi)))
            lo, end = bd.shard_read_range(text.size, m, lo, hi)
            shards.append(torch.from_numpy(text[lo:end].copy()).to(torch.device("cuda", r)))
            bases.append(lo)
        ptrs = (c_void_p * R)(*[t.data_ptr() for t in shards])
        ns = (c_int64 * R)(*[t.numel() for t in shards])
        bs = (c_int64 * R)(*bases)
        C = want.size
        for cap in sorted({C + 1, C, max(C - 1, 0), ends[0] + 1, 1, 0}, reverse=True):
            count, per = c_uint64(), (c_uint64 * R)()
            out = guarded(G + cap + G, "cuda:0")
            ok(bmx, lib.bmx_mg_search_device(mg._h, ptrs, ns, bs, pat, m, c_void_p(out.data_ptr() + 8 * G), cap,
                                             byref(count), per))
            torch.cuda.synchronize()
            assert count.value == C, (kind, cap, count.value, C)
            assert list(per) == [ends[0]] + [ends[r] - ends[r - 1] for r in range(1, R)], (kind, cap, list(per))
            buf = out.cpu().numpy()
            assert_same(buf, expect(buf.size, [(G, want[:cap])]), ("mg across calls", kind, cap))
    mg.close()


# ---------------------------------------------------------------------------------------------------------------
# 3. One process per GPU over cudaIpc mappings, a different step every time
# ---------------------------------------------------------------------------------------------------------------
IPC_STEPS, IPC_HEAD, IPC_TAIL, IPC_DEPTH = 9, 64, 1 << 14, 4


def _ipc_steps_worker(rank, world, port, seed, out_dir):
    import torch.distributed as dist

    import parallel_implementation_of_string_matching_algorithms_opencl_b200 as bmx
    from conftest import load_oracle
    from parallel_implementation_of_string_matching_algorithms_opencl_b200 import distributed as bd

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    steps = make_steps(load_oracle(), seed, world, IPC_DEPTH, IPC_STEPS)   # every rank builds the same steps
    x = bd.PeerExchange(dev, head_cap=IPC_HEAD, tail_cap=IPC_TAIL, depth=IPC_DEPTH)
    stream = torch.cuda.current_stream().cuda_stream
    sc = bmx.Scanner(dev.index)
    outs, keep, got = {}, {}, {}

    def post(q):
        st = steps[q - 1]
        a, b = st.read_range(rank)
        td = torch.from_numpy(st.text[a:b].copy()).to(dev)
        cap = max(st.counts[rank] + 5, 1)                  # lists that fit: the dense steps go through the tail
        pos = torch.empty(cap, dtype=torch.int64, device=dev)
        keep[q] = (td, pos)
        sc.set_pattern(st.pat, stream=stream)
        sc.begin(pos, stream=stream)
        cuts = st.pieces[rank] if st.shape[rank] == "normal" else [a, a]
        for k in range(max(len(cuts) - 1, 1)):
            lo, hi = cuts[k] - a, min(cuts[k + 1] + st.m - 1 - a, td.numel())
            sc.scan(td[lo:hi], cuts[k], stream=stream)
        x.post(sc, stream)

    def collect(q):
        outs[q] = torch.full((1 << 15,), -7, dtype=torch.int64, device=dev) if rank == 0 else None
        assert x.collect(outs[q], stream) == q
        total, counts, glen = x.wait(q)
        torch.cuda.synchronize()
        got[q] = (total, counts, None if outs[q] is None else outs[q][:glen].cpu().numpy())
        del keep[q], outs[q]

    for q in range(1, IPC_STEPS + 1):                     # bench.py's order: post q, then collect q-1
        post(q)
        if q > 1:
            collect(q - 1)
    collect(IPC_STEPS)
    np.save(os.path.join(out_dir, f"counts_{rank}.npy"), np.array([[t] + c for t, c, _ in (got[q] for q in sorted(got))], dtype=np.int64))
    if rank == 0:
        np.savez(os.path.join(out_dir, "gathered.npz"), **{f"s{q}": got[q][2] for q in got})
    dist.barrier()
    x.close()
    sc.close()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_exchange_processes_distinct_steps(bmx, oracle, tmp_path):
    """One process per GPU (up to 4), cudaIpc mappings, pipelined order, a different text and pattern every step."""
    import torch.multiprocessing as mp

    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs two GPUs")
    seed = 4242
    mp.spawn(_ipc_steps_worker, args=(world, _free_port(), seed, str(tmp_path)), nprocs=world, join=True)
    steps = make_steps(oracle, seed, world, IPC_DEPTH, IPC_STEPS)
    assert any(max(st.counts) > IPC_HEAD for st in steps)
    gathered = np.load(tmp_path / "gathered.npz")
    for r in range(world):
        rows = np.load(tmp_path / f"counts_{r}.npy")
        for q, st in enumerate(steps, 1):
            assert rows[q - 1][0] == st.truth.size and list(rows[q - 1][1:]) == st.counts, (r, q)
    for q, st in enumerate(steps, 1):
        held = [c + 5 for c in st.counts]
        k = sum(shipped(st.counts, held, IPC_HEAD + IPC_TAIL))
        assert gathered[f"s{q}"].size == k, ("ipc step", q, gathered[f"s{q}"].size, k)
        assert_same(gathered[f"s{q}"], st.truth[:k], ("ipc step", q))


# ---------------------------------------------------------------------------------------------------------------
# 4. combine_hits (the --exchange nccl path) returns the same prefix as the library exchange (CPU, gloo)
# ---------------------------------------------------------------------------------------------------------------
COMBINE_N, COMBINE_M, COMBINE_SEED = 40_009, 10, 31
FORMS = (("list", 4096), ("list", 3), ("packed", 4096), ("packed", 3))   # fast_cap above / below the held entries


def _combine_caps(world):
    """Per-rank caps (None: the whole list), capped below the count at different ranks."""
    if world == 2:
        return [(None, None), (5, None), (None, 5), (5, 5), (0, None), (2, 0)]
    return [(None, None, None), (None, 5, None), (None, None, 5), (5, None, 5), (None, 0, None), (2, 9, None)]


def _combine_text(bmx, world):
    from parallel_implementation_of_string_matching_algorithms_opencl_b200 import distributed as bd
    alpha = bmx.synth.ALPHABETS["dna"]
    pat = bmx.synth.pattern_from_stream(COMBINE_M, COMBINE_SEED, alpha)
    text = bmx.synth.fill_host(0, COMBINE_N, COMBINE_SEED, alpha)
    plants = list(bmx.synth.plant_offsets(COMBINE_N, COMBINE_M, 60, COMBINE_SEED))
    for r in range(1, world):
        seam, _ = bd.shard_bounds(COMBINE_N, world, r)
        plants += [seam - COMBINE_M // 2, seam - 1, seam]
    bmx.synth.plant_host(text, pat, [p for p in plants if 0 <= p <= COMBINE_N - COMBINE_M])
    return text, pat


def _combine_worker(rank, world, dst, port, out_dir):
    import torch.distributed as dist

    import parallel_implementation_of_string_matching_algorithms_opencl_b200 as bmx
    from conftest import load_oracle
    from parallel_implementation_of_string_matching_algorithms_opencl_b200 import distributed as bd

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    text, pat = _combine_text(bmx, world)
    lo, hi = bd.shard_bounds(COMBINE_N, world, rank)
    lo, end = bd.shard_read_range(COMBINE_N, COMBINE_M, lo, hi)
    mine = load_oracle().search(text[lo:end].tobytes(), pat) + lo      # the oracle plays the device
    res = {}
    for i, caps in enumerate(_combine_caps(world)):
        cap = caps[rank]
        pos = torch.from_numpy(mine[:cap].copy() if cap is not None else mine.copy())
        for form, fast_cap in FORMS:
            if form == "list":
                total, counts, gathered = bd.combine_hits(mine.size, pos, device=torch.device("cpu"), dst=dst,
                                                          fast_cap=fast_cap)
            else:
                packed = torch.zeros(2 + fast_cap, dtype=torch.int64)
                packed[0], packed[1] = mine.size, pos.numel()
                packed[2:2 + min(pos.numel(), fast_cap)] = pos[:fast_cap]
                total, counts, gathered = bd.combine_hits_start(None, pos, device=torch.device("cpu"), dst=dst,
                                                                fast_cap=fast_cap, packed=packed).finish()
            res[f"{i}-{form}-{fast_cap}-counts"] = np.array([total] + counts, dtype=np.int64)
            res[f"{i}-{form}-{fast_cap}-gathered"] = np.array([-1]) if gathered is None else gathered.numpy()
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), **res)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,dst", [(2, 0), (2, 1), (3, 0), (3, 2)])
def test_combine_hits_returns_the_library_prefix(world, dst, tmp_path, bmx, oracle):
    """Exact counts on every rank; on dst, whole lists in rank order up to and including the first rank whose list
    is capped below its count, nothing behind it -- with fast_cap above and below the held entries, and packed."""
    import torch.multiprocessing as mp
    from parallel_implementation_of_string_matching_algorithms_opencl_b200 import distributed as bd

    mp.spawn(_combine_worker, args=(world, dst, _free_port(), str(tmp_path)), nprocs=world, join=True)
    text, pat = _combine_text(bmx, world)
    want = kmp(oracle, text, pat)
    bounds = [bd.shard_bounds(COMBINE_N, world, r) for r in range(world)]
    counts = [int(((want >= lo) & (want < hi)).sum()) for lo, hi in bounds]
    assert min(counts) > 9, counts                                     # every cap below is below its rank's count
    got = [np.load(tmp_path / f"rank{r}.npz") for r in range(world)]
    for i, caps in enumerate(_combine_caps(world)):
        held = [c if cap is None else min(c, cap) for c, cap in zip(counts, caps)]
        prefix = want[:sum(shipped(counts, held, 1 << 62))]
        for form, fast_cap in FORMS:
            tag = f"{i}-{form}-{fast_cap}"
            for r in range(world):
                assert list(got[r][f"{tag}-counts"]) == [want.size] + counts, (tag, r)
                if r != dst:
                    assert list(got[r][f"{tag}-gathered"]) == [-1], (tag, r)
            g = got[dst][f"{tag}-gathered"]
            assert g.size == prefix.size, (tag, caps, "gathered", g.tolist(), "want a prefix of", prefix.size)
            assert_same(g, prefix, (tag, caps))
