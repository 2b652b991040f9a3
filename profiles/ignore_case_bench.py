#!/usr/bin/env python
"""Case-insensitive search (BMX_IGNORE_CASE) against the exact search and against what a user does without it.

Three arms per workload, alternated run by run in one process, each timed with CUDA events around the device work:
  exact      the exact search (bmx_scanner_begin + bmx_scanner_scan), the rate reference;
  icase      the case-insensitive search of a mixed-case pattern on the same text;
  lower+ex   a lowered device copy of the text (one torch expression) followed by the exact search of the lowered
             pattern, timed together.
Positions and count-only, median of --runs warmed runs.  icase and lower+ex must agree on the count and the list.
Workloads: 4 GiB DNA m = 32, 4 GiB ascii95 m = 16, 4 GiB bytes256 m = 4 (WINDOW, a letter pattern), and the English
fixture (input5L) tiled to 1 GiB with five patterns.

python profiles/ignore_case_bench.py --out profiles/ignore_case_bench.txt"""
from __future__ import annotations

import argparse
import statistics
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

GIB = 1 << 30


def mixcase(pat: bytes, seed: int) -> bytes:
    rng = np.random.default_rng(seed)
    flip = rng.integers(0, 2, size=len(pat)).astype(bool)
    out = bytes(c ^ 0x20 if f and chr(c).isascii() and chr(c).isalpha() else c for c, f in zip(pat, flip))
    return out if out != pat or not any(chr(c).isalpha() for c in pat) else out.swapcase()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=25)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

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
    out(f"# card: {torch.cuda.get_device_name(0)} | nvidia-smi name, power limit, max SM clock: "
        f"{q.stdout.strip().splitlines()[0] if q.stdout else 'n/a'}")
    out(f"# {a.runs} warmed runs per arm, arms alternated run by run; median device-event time; GB/s = text bytes / time")
    out("# lower+ex = torch.where((t >= 65) & (t <= 90), t + 32, t) into a new tensor, then the exact search, timed together")
    stream = torch.cuda.current_stream(dev)
    sh = stream.cuda_stream
    scanners = {arm: bmx.Scanner(0) for arm in ("exact", "icase", "lower+ex")}
    for sc in scanners.values():
        sc.set_timing(0)

    def lower(t):
        return torch.where((t >= 65) & (t <= 90), t + 32, t)

    def workload(name, text, pats, variant="auto"):
        n = text.numel()
        pos = {arm: torch.empty(max(n // 16, 1 << 20), dtype=torch.int64, device=dev) for arm in scanners}
        for pat_exact, pat_ic in pats:
            scanners["exact"].set_pattern(pat_exact, variant=variant, stream=sh)
            scanners["icase"].set_pattern(pat_ic, variant=variant, stream=sh, ignore_case=True)
            scanners["lower+ex"].set_pattern(pat_ic.lower(), variant=variant, stream=sh)
            for mode in ("positions", "count"):
                def run(arm):
                    sc = scanners[arm]
                    src = lower(text) if arm == "lower+ex" else text
                    sc.begin(pos[arm] if mode == "positions" else None, stream=sh)
                    sc.scan(src, 0, stream=sh)
                    return src
                times = {arm: [] for arm in scanners}
                counts, stats = {}, {}
                for r in range(a.runs + 3):
                    for arm in scanners:
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record(stream)
                        src = run(arm)
                        e1.record(stream)
                        counts[arm], stats[arm] = scanners[arm].finish(stream=sh)
                        del src
                        if r >= 3:
                            times[arm].append(e0.elapsed_time(e1))
                assert stats["icase"]["ignore_case"] and not stats["exact"]["ignore_case"]
                ok = counts["icase"] == counts["lower+ex"]
                if mode == "positions":
                    k = min(counts["icase"], pos["icase"].numel())
                    ok = ok and bool(torch.equal(pos["icase"][:k], pos["lower+ex"][:k]))
                med = {arm: statistics.median(v) for arm, v in times.items()}
                gbs = {arm: n / (ms * 1e-3) / 1e9 for arm, ms in med.items()}
                out(f"{name:18s} {pat_ic.decode('latin-1')!r:30s} {mode:9s} "
                    f"exact {gbs['exact']:7.0f}  icase {gbs['icase']:7.0f}  lower+ex {gbs['lower+ex']:6.0f} GB/s  "
                    f"icase/exact {gbs['icase'] / gbs['exact']:5.3f}  icase vs lower+ex {med['lower+ex'] / med['icase']:5.1f}x  "
                    f"hits exact {counts['exact']} icase {counts['icase']}  same-as-lower+ex {ok}")
                assert ok, (name, pat_ic, mode)
        del pos

    out(f"{'workload':18s} {'pattern (icase arm)':30s} {'mode':9s}")
    # ---- synthetic 4 GiB texts
    for name, alpha_key, m, variant, pat in (("dna 4GiB", "dna", 32, "auto", None), ("ascii95 4GiB", "ascii95", 16, "auto", None),
                                             ("bytes256 4GiB", "bytes256", 4, "window", b"KiNg")):
        alpha = bmx.synth.ALPHABETS[alpha_key]
        text = torch.empty(4 * GIB, dtype=torch.uint8, device=dev)
        bmx.synth.fill_device(text, 0, 17, alpha)
        if pat is None:
            pat = bmx.synth.pattern_from_stream(m, 17, alpha)
            if not any(chr(c).isalpha() for c in pat):
                pat = b"Q" + pat[1:]
        bmx.synth.plant_device(text, pat, bmx.synth.plant_offsets(text.numel(), m, 2000, 17))
        pat_ic = pat.lower() if alpha_key == "dna" else mixcase(pat, m)
        workload(name, text, [(pat, pat_ic)], variant)
        del text
        torch.cuda.empty_cache()

    # ---- the English fixture tiled to 1 GiB
    base = np.frombuffer(Golden(ROOT / "tests" / "golden" / "golden.npz").text("input5L"), dtype=np.uint8)
    text = torch.from_numpy(np.tile(base, GIB // base.size + 1)[:GIB].copy()).to(dev)
    pats = [(p, mixcase(p, len(p))) for p in (b"is", b"the", b"position", b"HACKHACK", b"occurrences starting from")]
    workload("english 1GiB", text, pats)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
