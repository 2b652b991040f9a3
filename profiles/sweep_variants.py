#!/usr/bin/env python
"""Measures every scan variant per (alphabet, pattern length) on one B200 and writes
profiles/variants_<tag>.json -- the table that justifies the variant thresholds of bmx::choose_filter()
(north star: "chosen per pattern length and justified by measurement").

    python profiles/sweep_variants.py --tag r01 [--gib 1] [--steps 10]

Device-resident text, positions written, CUDA-event timed, K back-to-back scans per cell.
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

import parallel_implementation_of_string_matching_algorithms_opencl_b200 as bmx  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", default="r01")
    ap.add_argument("--gib", type=float, default=1.0)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    n = int(args.gib * (1 << 30))
    stream = torch.cuda.current_stream().cuda_stream
    scanner = bmx.Scanner(0)
    pos = torch.empty(1 << 20, dtype=torch.int64, device=dev)
    rows = []
    for alpha_name in ("dna", "ascii95", "bytes256"):
        alpha = bmx.synth.ALPHABETS[alpha_name]
        text = torch.empty(n, dtype=torch.uint8, device=dev)
        bmx.synth.fill_device(text, 0, 1234, alpha)
        for m in (1, 2, 3, 4, 5, 6, 7, 8, 10, 11, 12, 16, 24, 32, 33, 64, 128):
            if alpha_name == "dna" and m < 8:
                continue  # millions of natural hits: an output benchmark, not a filter benchmark
            if alpha_name == "ascii95" and m < 3:
                continue
            pat = bmx.synth.pattern_from_stream(m, 1000 + m, alpha)
            bmx.synth.plant_device(text, pat, bmx.synth.plant_offsets(n, m, 100, m))
            torch.cuda.synchronize()
            cell = {"alphabet": alpha_name, "m": m, "n": n}
            counts = set()
            for variant in ("window", "qgram", "shiftand"):
                if (variant == "qgram" and m < 7) or (variant == "shiftand" and m > 32):
                    continue
                scanner.set_pattern(pat, variant=variant, stream=stream)
                for _ in range(3):
                    scanner.begin(pos, stream=stream)
                    scanner.scan(text, 0, stream=stream)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    scanner.begin(pos, stream=stream)
                    scanner.scan(text, 0, stream=stream)
                e1.record()
                torch.cuda.synchronize()
                count, _ = scanner.finish(stream=stream)
                counts.add(count)
                cell[variant] = round(n / (e0.elapsed_time(e1) / args.steps * 1e-3) / 1e9, 1)
            cell["hits"] = counts.pop() if len(counts) == 1 else f"MISMATCH {sorted(counts)}"
            cell["auto"] = bmx._lib.VARIANT_NAMES[bmx._lib.load().bmx_version() and (1 if m >= 7 else 2)]
            rows.append(cell)
            print(cell, flush=True)
        del text
    out = Path(args.out) if args.out else ROOT / "profiles" / f"variants_{args.tag}.json"
    out.write_text(json.dumps({"unit": "GB/s of text scanned, positions written, device-timed", "rows": rows}, indent=1))
    print("wrote", out)


if __name__ == "__main__":
    main()
