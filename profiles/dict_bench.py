#!/usr/bin/env python
"""Dictionary search (bmx_dict_search_device) over device-resident text larger than L2: one pass for K patterns,
counts only and with (position, pattern) pairs, against one single-pattern pass (K passes cost K times that) and
against bmx_search_multi_device at K = 64.  Times are CUDA-event medians of warmed calls; the card's name and power
limit are read in the same run.  Counts are checked against single-pattern searches for a sample of patterns.
    python profiles/dict_bench.py [--gib 4] [--reps 5] [--ks 64,256,...]"""
from __future__ import annotations

import argparse
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import parallel_implementation_of_string_matching_algorithms_opencl_b200 as bmx  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--gib", type=float, default=4.0)
ap.add_argument("--english-gib", type=float, default=1.0)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--ks", default="64,256,1024,4096,16384,65536")
args = ap.parse_args()
KS = [int(k) for k in args.ks.split(",")]
dev = torch.device("cuda:0")


def median_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times), r


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def run(label, text, patterns_for, m):
    n = text.numel()
    one_ms, _ = median_ms(lambda: bmx.search_device(text, patterns_for(1)[0], timing=False), args.reps)
    print(f"{label}: n={n / 2**30:.2f} GiB m={m}  single-pattern pass {one_ms:.3f} ms", flush=True)
    for K in KS:
        pats = patterns_for(K)
        d = bmx.Dictionary(pats)
        c_ms, (counts, _, _, total) = median_ms(lambda: d.search_device(text), args.reps)
        p_ms, (_, pos, _, ptotal) = median_ms(lambda: d.search_device(text, max_matches=1 << 20), args.reps)
        assert ptotal == total
        line = (f"  K={K:<6d} counts {c_ms:8.3f} ms ({n / c_ms / 1e6:7.1f} GB/s)   pairs {p_ms:8.3f} ms   "
                f"K passes ~{K * one_ms:9.1f} ms (x{K * one_ms / c_ms:7.1f})   pairs {total}")
        if K == 64:
            m_ms, res = median_ms(lambda: bmx.search_multi_device(text, pats, max_positions=4096), args.reps)
            assert [c for c, _ in res] == [int(c) for c in counts]
            line += f"   search_multi {m_ms:.3f} ms"
        print(line, flush=True)
        rng = np.random.default_rng(K)
        for k in rng.choice(K, size=min(K, 3), replace=False):
            assert bmx.search_device(text, pats[k], timing=False)[0] == int(counts[k]), (label, K, k)
        d.close()


print(f"card: {card()}", flush=True)
n = int(args.gib * 2**30)
for alphabet, m in (("dna", 32), ("ascii95", 16), ("bytes256", 8)):
    alpha = bmx.synth.ALPHABETS[alphabet]
    text = torch.empty(n, dtype=torch.uint8, device=dev)
    bmx.synth.fill_device(text, 0, 43, alpha)
    cut = lambda K, alpha=alpha, m=m: [bmx.synth.fill_host(1_000_003 * (k + 1) % (n - m), m, 43, alpha).tobytes()  # noqa: E731
                                       for k in range(K)]   # cut from the text: sparse, >= 1 hit each
    run(f"{alphabet}", text, cut, m)
    del text
    torch.cuda.empty_cache()

# English: the reference's fixture tiled to the requested size, its own words of >= 7 bytes (then random 7..16-byte
# strings of its letters to reach K)
z = np.load(ROOT / "tests" / "golden" / "golden.npz")
eng = bytes(z["text/input5L"])
words = sorted({w for w in eng.split() if len(w) >= 7})
rng = np.random.default_rng(7)
letters = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz", dtype=np.uint8)
extra = [letters[rng.integers(0, 26, size=int(rng.integers(7, 17)))].tobytes() for _ in range(max(KS))]
ne = int(args.english_gib * 2**30)
base = torch.from_numpy(np.frombuffer(eng, dtype=np.uint8).copy()).to(dev)
text = base.repeat(ne // base.numel() + 1)[:ne].contiguous()
run(f"english ({len(words)} words >= 7 bytes)", text, lambda K: (words + extra)[:K], 7)
