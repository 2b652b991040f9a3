#!/usr/bin/env python
"""Many ranges in one call (bmx_search_ranges[_device]) against one positions scan of the same bytes, against a
per-document loop, and the partition mirror (bmx_search_partitions) of this library against another build.

  1. bmx_search_ranges_device over 1 GiB (device-resident) cut into D = 1, 10^3, 10^6, 10^7 random documents, sparse
     DNA m = 32 and the English fixture tiled to 1 GiB ("is"); beside it bmx_search_device over the same 1 GiB with
     positions.  Times: host clock around the synchronous C call, median of --reps after two warm-up calls.
  2. us per document: bmx_search_device on each of the first 10^4 documents of the D = 10^6 cut, against the batch.
  3. bmx_search_partitions on the reference's 500 KB fixture, P = 2, 1000, 10000 words ranges; with --old LIB the same
     in a child process bound to that build (BMX_LIB), so both columns come from the same box.
  4. bmx_search_ranges (host entry) over both corpora from pinned host memory, against bmx_search_ex on the same bytes.
Every batched result is checked against the plain scan's list (np.searchsorted) before it is timed.
Usage: python profiles/ranges_bench.py [--old other_libbmx.so] [--reps 20] [--out FILE]"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import time
from ctypes import c_int64, c_uint64, c_void_p
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

GIB = 1 << 30


def median_ms(fn, reps: int) -> float:
    fn()
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def partitions_rows(reps: int) -> list:
    """[{P, us per call, total}] of bmx_search_partitions on input5L, pattern "is", in the build BMX_LIB names (the
    binding is made here, so that a build without the newer entry points loads as well)."""
    from conftest import Golden

    text = Golden(ROOT / "tests" / "golden" / "golden.npz").text("input5L")
    so = os.environ.get("BMX_LIB") or str(ROOT / "parallel_implementation_of_string_matching_algorithms_opencl_b200" / "libbmx.so")
    lib = ctypes.CDLL(so)
    p32 = ctypes.POINTER(ctypes.c_int32)
    lib.bmx_partition_words.argtypes = [c_void_p, c_int64, ctypes.c_int32, p32]
    lib.bmx_search_partitions.argtypes = [c_void_p, ctypes.c_char_p, p32, p32, p32, p32, ctypes.c_int32, ctypes.c_int32]
    buf = np.frombuffer(text, dtype=np.uint8)
    rows = []
    for P in (2, 1000, 10_000):
        se = np.zeros(2 * P, dtype=np.int32)
        assert lib.bmx_partition_words(buf.ctypes.data, buf.size, P, se.ctypes.data_as(p32)) == 0
        ans = np.zeros(P, dtype=np.int32)

        def call():
            rc = lib.bmx_search_partitions(buf.ctypes.data, b"is", se.ctypes.data_as(p32), ans.ctypes.data_as(p32), None, None, 2, P)
            assert rc == 0, rc
        us = median_ms(call, reps if P < 10_000 else max(3, reps // 4)) * 1e3
        rows.append({"P": P, "us": round(us, 1), "total": int(ans.sum())})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--old", default="", help="another build of libbmx.so for the partition-mirror column")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    ap.add_argument("--partitions-only", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.partitions_only:
        print(json.dumps(partitions_rows(a.reps)))
        return

    import torch

    import parallel_implementation_of_string_matching_algorithms_opencl_b200 as bmx
    from conftest import Golden

    lines = []

    def out(s=""):
        print(s, flush=True)
        lines.append(s)

    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    out(f"# card: {torch.cuda.get_device_name(0)} | nvidia-smi: {q.stdout.strip().splitlines()[0] if q.stdout else 'n/a'}")
    out(f"# library: {Path(bmx.LIB_PATH).resolve().relative_to(ROOT) if Path(bmx.LIB_PATH).resolve().is_relative_to(ROOT) else Path(bmx.LIB_PATH).name}; reps {a.reps}, median; host clock around each synchronous call")
    lib = bmx._lib.load()
    stream = torch.cuda.current_stream(dev)
    st = c_void_p(stream.cuda_stream)

    # ---- corpora, 1 GiB each, device-resident
    alpha = bmx.synth.ALPHABETS["dna"]
    dna = torch.empty(GIB, dtype=torch.uint8, device=dev)
    bmx.synth.fill_device(dna, 0, 31, alpha)
    pat_dna = bmx.synth.pattern_from_stream(32, 31, alpha)
    bmx.synth.plant_device(dna, pat_dna, bmx.synth.plant_offsets(GIB, 32, 1000, 31))
    eng = Golden(ROOT / "tests" / "golden" / "golden.npz").text("input5L")
    reps_eng = GIB // len(eng) + 1
    english = torch.from_numpy(np.frombuffer(eng * reps_eng, dtype=np.uint8)[:GIB].copy()).to(dev)
    corpora = [("dna m=32", dna, pat_dna), ("english 'is'", english, b"is")]

    rng = np.random.default_rng(5)
    cuts = {}
    for D in (1, 1000, 10**6, 10**7):
        c = np.sort(rng.integers(1, GIB, D - 1))   # repeated cuts make empty documents, which are allowed
        cuts[D] = torch.as_tensor(np.concatenate([[0], c, [GIB]]).astype(np.int64), device=dev)

    out("\n## 1. one call over 1 GiB cut into D documents (device entry) vs one positions scan of the 1 GiB")
    out(f"{'corpus':<14} {'D':>9} {'hits':>10} {'scan ms':>8} {'ranges ms':>10} {'ratio':>6} {'ns/doc':>8}")
    batched_per_doc = {}
    for name, t, pat in corpora:
        cnt = c_uint64(0)
        pos = torch.empty(GIB // 16, dtype=torch.int64, device=dev)
        def scan():
            bmx._lib.check(lib.bmx_search_device(c_void_p(t.data_ptr()), GIB, pat, len(pat), c_void_p(pos.data_ptr()), pos.numel(),
                                                 ctypes.byref(cnt), None, st))
        scan_ms = median_ms(scan, a.reps)
        hits = cnt.value
        whole = pos[:hits].cpu().numpy()
        for D, offs in cuts.items():
            counts = torch.empty(D, dtype=torch.int64, device=dev)
            offsets = torch.empty(D + 1, dtype=torch.int64, device=dev)
            rpos = torch.empty(max(hits, 1), dtype=torch.int64, device=dev)
            total = c_uint64(0)
            b, e = offs[:-1], offs[1:]
            def ranges():
                bmx._lib.check(lib.bmx_search_ranges_device(c_void_p(t.data_ptr()), GIB, D, c_void_p(b.data_ptr()), c_void_p(e.data_ptr()),
                                                            pat, len(pat), c_void_p(rpos.data_ptr()), rpos.numel(),
                                                            c_void_p(counts.data_ptr()), c_void_p(offsets.data_ptr()),
                                                            ctypes.byref(total), st))
            ranges()
            # correctness before timing: the per-document counts follow from the whole list
            bn, en = b.cpu().numpy(), e.cpu().numpy()
            want = np.searchsorted(whole, en - len(pat) + 1) - np.searchsorted(whole, bn)
            want = np.where(en - bn >= len(pat), want, 0)
            assert np.array_equal(counts.cpu().numpy(), want), (name, D)
            assert total.value == int(want.sum()) <= hits
            ms = median_ms(ranges, a.reps)
            batched_per_doc[(name, D)] = ms * 1e6 / D
            out(f"{name:<14} {D:>9} {total.value:>10} {scan_ms:>8.3f} {ms:>10.3f} {ms / scan_ms:>6.2f} {ms * 1e6 / D:>8.1f}")
            del counts, offsets, rpos
        del pos
        torch.cuda.empty_cache()

    out("\n## 2. per-document loop of bmx_search_device (first 10^4 documents of the D = 10^6 cut) vs the batched call")
    out(f"{'corpus':<14} {'loop us/doc':>12} {'batched us/doc':>15} {'ratio':>8}")
    offs = cuts[10**6].cpu().numpy()
    for name, t, pat in corpora:
        pos = torch.empty(1 << 16, dtype=torch.int64, device=dev)
        cnt = c_uint64(0)
        docs = [(int(offs[i]), int(offs[i + 1])) for i in range(10_000)]
        def loop():
            for lo, hi in docs:
                bmx._lib.check(lib.bmx_search_device(c_void_p(t.data_ptr() + lo), hi - lo, pat, len(pat), c_void_p(pos.data_ptr()),
                                                     pos.numel(), ctypes.byref(cnt), None, st))
        loop_us = median_ms(loop, 3) * 1e3 / len(docs)
        per = batched_per_doc[(name, 10**6)] / 1e3
        out(f"{name:<14} {loop_us:>12.2f} {per:>15.4f} {loop_us / per:>8.0f}")

    out("\n## 3. bmx_search_partitions, reference fixture input5L (500 KB), pattern 'is', us per call")
    new = partitions_rows(a.reps)
    old = None
    if a.old:
        env = dict(os.environ, BMX_LIB=str(Path(a.old).resolve()))
        r = subprocess.run([sys.executable, __file__, "--partitions-only", "--reps", str(a.reps)], env=env,
                           capture_output=True, text=True, check=True)
        old = json.loads(r.stdout.strip().splitlines()[-1])
    out(f"{'P':>6} {'this library':>13} {'other build':>12} {'same totals':>12}")
    for i, row in enumerate(new):
        o = old[i] if old else None
        out(f"{row['P']:>6} {row['us']:>13.1f} {(o['us'] if o else float('nan')):>12.1f} {str(o['total'] == row['total']) if o else '-':>12}")

    out("\n## 4. host entry end to end from pinned memory: bmx_search_ranges vs bmx_search_ex over the same 1 GiB")
    out(f"{'corpus':<14} {'D':>9} {'search_ex ms':>13} {'ranges ms':>10} {'ratio':>6}")
    for name, t, pat in corpora:
        host = torch.empty(GIB, dtype=torch.uint8, pin_memory=True)
        host.copy_(t.cpu())
        cnt = c_uint64(0)
        hpos = np.empty(GIB // 16, dtype=np.int64)
        def plain():
            bmx._lib.check(lib.bmx_search_ex(0, c_void_p(host.data_ptr()), GIB, pat, len(pat), hpos.ctypes.data, hpos.size,
                                             ctypes.byref(cnt), 0, None))
        plain_ms = median_ms(plain, 5)
        for D in (1000, 10**6):
            o = cuts[D].cpu().numpy()
            b, e = np.ascontiguousarray(o[:-1]), np.ascontiguousarray(o[1:])
            counts = np.zeros(D, dtype=np.uint64)
            offsets = np.zeros(D + 1, dtype=np.int64)
            def ranges():
                bmx._lib.check(lib.bmx_search_ranges(0, c_void_p(host.data_ptr()), GIB, D, b.ctypes.data, e.ctypes.data, pat, len(pat),
                                                     hpos.ctypes.data, hpos.size, counts.ctypes.data, offsets.ctypes.data))
            ranges()
            assert int(offsets[-1]) <= cnt.value and np.array_equal(np.cumsum(counts.astype(np.int64)), offsets[1:])
            ms = median_ms(ranges, 5)
            out(f"{name:<14} {D:>9} {plain_ms:>13.2f} {ms:>10.2f} {ms / plain_ms:>6.2f}")
        del host

    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
