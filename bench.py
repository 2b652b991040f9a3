#!/usr/bin/env python
"""bench.py -- text GB/s scanned by the Boyer-Moore path on B200 (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one batch of synthetic text:
  N = 1   workload dna_m32_4GiB      (BASELINE.json configs[1]: 4 GiB random DNA, m = 32)
  N > 1   workload ascii95_m64_shard (configs[4]: 8 GiB per GPU of 95-symbol ASCII, m = 64,
                                      sharded with (m-1) halo, counts and position
                                      lists gathered to rank 0 over NCCL) -- weak scaling.
`value`  : device-resident text, CUDA-event timed, K back-to-back scans (positions written).
`e2e`    : the same scan through the host-pointer C-ABI call bmx_search_ex: pinned host text,
           host->device copy, scan and position read-back all inside the timed region.
`roofline`: algorithmic bytes (n + 8*hits) per scan-kernel launch / its average duration vs the
           measured HBM copy bandwidth of MEASURED_PEAKS.json.
`cpu_baseline`: the reference's own serial code (oracle/_ref/libref_bm.so, 1 core) on a bounded
           sample of the same text (rank 0, N = 1 only).
--impl reference: the reference's own CPU code on all host threads (windowed), same metric.
--dump-outputs DIR: what the last timed step returned (on rank 0: the match count and the ascending
           start positions) as DIR/count.npy, DIR/positions.npy and DIR/positions_index.npy, float64.
           The inputs are fixed by the workload's seeds, so two builds can be compared file by file.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

GIB = 1 << 30
_REAL_STDOUT = None


def emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)
WORKLOADS = {
    # name: (alphabet, bytes per GPU, m, seed, plants per GPU, pattern source)
    "dna_m32_4GiB": dict(alphabet="dna", n=4 * GIB, m=32, seed=43, plants=1000, pattern="from_text"),
    "ascii95_m64_shard": dict(alphabet="ascii95", n=8 * GIB, m=64, seed=47, plants=1000, pattern="random"),
    "ascii95_m16_64MiB": dict(alphabet="ascii95", n=64 << 20, m=16, seed=42, plants=1000, pattern="random"),
    "bytes256_m4_4GiB": dict(alphabet="bytes256", n=4 * GIB, m=4, seed=44, plants=1000, pattern="random"),
    "bytes256_m16_4GiB": dict(alphabet="bytes256", n=4 * GIB, m=16, seed=45, plants=1000, pattern="random"),
    "bytes256_m128_4GiB": dict(alphabet="bytes256", n=4 * GIB, m=128, seed=46, plants=1000, pattern="random"),
    "aaa_1GiB": dict(alphabet="a", n=1 * GIB, m=3, seed=1, plants=0, pattern="aaa"),
    # not BASELINE configs: the reference's own kind of input at scale (its English fixture input5L.txt, from
    # tests/golden/golden.npz, tiled to 1 GiB; its own query "is" and a phrase of its console output) and the weakest
    # sparse case (short pattern, 4-letter alphabet).  Reported in `configs` with "baseline_config": false.
    "english_is_1GiB": dict(alphabet="english", n=1 * GIB, m=2, seed=0, plants=0, pattern="is"),
    "english_m25_1GiB": dict(alphabet="english", n=1 * GIB, m=25, seed=0, plants=0, pattern="occurrences starting from"),
    "dna_m8_1GiB": dict(alphabet="dna", n=1 * GIB, m=8, seed=4321, plants=100, pattern="random"),
}
EXTRA_CONFIGS = ("english_is_1GiB", "english_m25_1GiB", "dna_m8_1GiB")


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._armed = False
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        if self.nv:
            try:   # the first queries of a process are slow (tens of ms): take them before the timed region
                self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                get = getattr(self.nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or self.nv.nvmlDeviceGetCurrentClocksThrottleReasons
                get(self.h)
            except Exception:
                pass

    def _run(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
        }
        while not self._stop.is_set():
            if not self._armed:          # started before the barrier (NVML set-up costs milliseconds), sampling only the timed region
                time.sleep(0.0002)
                continue
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                r = get(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.0005)

    def __enter__(self):
        if self.nv:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def arm(self):
        self._armed = True

    def __exit__(self, *a):
        self._stop.set()
        if self._thread:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def make_pattern(bmx, w, total_n):
    alpha = bmx.synth.ALPHABETS[w["alphabet"]]
    if w["pattern"] == "from_text":       # cut from the text itself (so there is at least one hit)
        off = bmx.synth.mix64(w["seed"] * 7919) % (total_n - w["m"])
        return bmx.synth.fill_host(off, w["m"], w["seed"], alpha).tobytes()
    if w["pattern"] == "random":
        return bmx.synth.pattern_from_stream(w["m"], w["seed"], alpha)
    return w["pattern"].encode()


def plant_list(bmx, w, total_n, world):
    """Global plant offsets: `plants` per GPU anywhere, plus plants straddling every shard seam."""
    from parallel_implementation_of_string_matching_algorithms_opencl_b200.distributed import shard_bounds
    offs = list(bmx.synth.plant_offsets(total_n, w["m"], w["plants"] * world, w["seed"]))
    if w["plants"]:
        for r in range(1, world):
            seam, _ = shard_bounds(total_n, world, r)
            for d in (w["m"] // 2, 1, w["m"] - 1):
                offs.append(seam - d)       # starts left of the seam, ends right of it
            offs.append(seam)
    return np.array(sorted(set(int(o) for o in offs if 0 <= o <= total_n - w["m"])), dtype=np.int64)


def verify_hits(torch, text, lo, pat, pos, count, cap):
    """Size-independent checks: ascending, every reported start really matches."""
    if count == 0 or pos is None:
        return True
    k = min(count, cap)
    p = pos[:k]
    ok = bool((p[1:] > p[:-1]).all().item()) if k > 1 else True
    sample = p if k <= 100000 else p[torch.randint(0, k, (100000,), device=p.device)]
    pt = torch.frombuffer(bytearray(pat), dtype=torch.uint8).to(text.device)
    idx = (sample - lo).unsqueeze(1) + torch.arange(len(pat), device=text.device).unsqueeze(0)
    ok = ok and bool((text[idx] == pt.unsqueeze(0)).all().item())
    return ok


DUMP_MAX_POSITIONS = 1 << 21     # positions + their indices, float64: 32 MiB per dump


def dump_outputs(torch, out_dir, count, positions):
    """Writes the result of one step as float64 arrays (exact for every position below 2^53): count.npy holds
    the match count, positions.npy the ascending start positions and positions_index.npy their indices in
    the full list.  A list longer than DUMP_MAX_POSITIONS is sampled at indices drawn from a fixed seed."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    held = 0 if positions is None else int(positions.numel())
    idx = np.arange(held)
    if held > DUMP_MAX_POSITIONS:
        idx = np.sort(np.random.default_rng(0).choice(held, DUMP_MAX_POSITIONS, replace=False))
        positions = positions[torch.from_numpy(idx).to(positions.device)]
    vals = positions.cpu().numpy() if held else np.zeros(0)
    np.save(out / "count.npy", np.array([count], dtype=np.float64))
    np.save(out / "positions.npy", vals.astype(np.float64))
    np.save(out / "positions_index.npy", idx.astype(np.float64))


def oracle_lib():
    """(library, function, kind-chooser) of the CPU checker: the reference's own code where its domain allows
    (7-bit bytes, m <= 99: oracle/_ref/libref_bm.so), else the widened restatement (oracle/liboracle.so)."""
    so = ROOT / "oracle" / "liboracle.so"
    if not so.exists():
        import subprocess
        subprocess.run(["bash", str(ROOT / "oracle" / "build_oracle.sh")], check=True, capture_output=True)
    port = ctypes.CDLL(str(so))
    ref_so = ROOT / "oracle" / "_ref" / "libref_bm.so"
    ref = ctypes.CDLL(str(ref_so)) if ref_so.exists() else None
    return port, ref


def oracle_search(arr, pat, want_positions: bool, threads: int = -1, cap_hint: int = 0):
    """CPU truth for a host uint8 array: (count, positions or None, kind).  All host threads, windowed."""
    port, ref = oracle_lib()
    n = int(arr.size)
    legal7 = len(pat) <= 99 and max(pat) < 0x80 and (n == 0 or int(arr[: min(n, 1 << 24)].max()) < 0x80)
    fn, kind = (ref.ref_bm_search_windowed, "reference") if (ref is not None and legal7) else (port.oracle_search_mt, "port")
    cnt = ctypes.c_uint64()
    cap = int(cap_hint) if want_positions else 0
    pos = np.empty(max(cap, 1), dtype=np.int64) if want_positions else None
    rc = fn(ctypes.c_void_p(arr.ctypes.data), ctypes.c_int64(n), ctypes.c_char_p(pat), ctypes.c_int32(len(pat)),
            ctypes.c_void_p(pos.ctypes.data) if want_positions else None, ctypes.c_int64(cap), ctypes.byref(cnt), ctypes.c_int32(threads))
    assert rc == 0, rc
    return int(cnt.value), (pos[: min(int(cnt.value), cap)] if want_positions else None), kind


def oracle_verdict(torch, text, lo, pat, count, pos, cap, dense, host=None):
    """The CUDA result against the oracle on the same bytes (outside every timed region): the shard goes back
    to the host, the reference's serial code (windowed over all host threads) scans it, and count + position
    list must be identical.  Dense texts (a list of ~n positions would need 8n bytes of host memory) compare
    the count with the oracle's and the list with its closed form on the device."""
    if host is None:
        host = text.cpu().numpy()
    if dense:
        ocount, _, kind = oracle_search(host, pat, False)
        k = min(count, cap)
        closed = bool((pos[:k] == torch.arange(lo, lo + k, device=pos.device, dtype=torch.int64)).all().item()) if k else True
        return bool(ocount == count and closed and count == host.size - len(pat) + 1), f"{kind}: count + closed-form list", ocount, None
    ocount, opos, kind = oracle_search(host, pat, True, cap_hint=max(count, 0) + 1024)
    got = pos[: min(count, cap)].cpu().numpy() - lo if pos is not None else np.zeros(0, dtype=np.int64)
    ok = ocount == count and (count > cap or np.array_equal(got, opos)) and np.array_equal(got, opos[: got.size])
    return bool(ok), f"{kind}: count + full position list", ocount, opos


def build_workload(bmx, torch, name, world, rank, dev, bytes_per_gpu=0):
    """Materialises this rank's shard of a named workload on the device."""
    from parallel_implementation_of_string_matching_algorithms_opencl_b200 import distributed as bd
    w = dict(WORKLOADS[name])
    if bytes_per_gpu:
        w["n"] = bytes_per_gpu
    if w["alphabet"] == "english":      # single GPU only: the reference's fixture tiled
        z = np.load(ROOT / "tests" / "golden" / "golden.npz")
        base = np.asarray(z["text/input5L"], dtype=np.uint8)
        n = w["n"]
        text = torch.from_numpy(np.tile(base, n // base.size + 1)[:n].copy()).to(dev)
        pat = w["pattern"].encode()
        return dict(name=name, w=w, m=len(pat), total_n=n, lo=0, end=n, pat=pat, plants=np.zeros(0, dtype=np.int64), text=text,
                    dense=False, cap=n // 8)
    alpha = bmx.synth.ALPHABETS[w["alphabet"]]
    m = w["m"]
    total_n = w["n"] * world
    lo, hi = bd.shard_bounds(total_n, world, rank)
    lo, end = bd.shard_read_range(total_n, m, lo, hi)
    pat = make_pattern(bmx, w, total_n)
    plants = plant_list(bmx, w, total_n, world)
    text = torch.empty(end - lo, dtype=torch.uint8, device=dev)
    bmx.synth.fill_device(text, lo, w["seed"], alpha)
    mine = plants[(plants + m > lo) & (plants < end)]
    bmx.synth.plant_device(text, pat, mine, base=lo)
    torch.cuda.synchronize()
    dense = w["alphabet"] == "a"
    cap = (end - lo) if dense else max(4 * len(plants) + 1024, 1 << 16)
    return dict(name=name, w=w, m=m, total_n=total_n, lo=lo, end=end, pat=pat, plants=plants, text=text, dense=dense, cap=cap)


def kernel_roofline(W, count, scan_ms, step_gpu_ms, peak):
    """Roofline record of the dominant kernel of one step (scan_kernel; expand_kernel when the text is dense)."""
    n = W["end"] - W["lo"]
    held = min(count, W["cap"])
    kernel_ms = (step_gpu_ms - scan_ms) if W["dense"] else scan_ms
    alg_bytes = 8 * held if W["dense"] else n      # expand writes the positions; scan reads the text
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    step_bytes = n + 8 * held
    return {"achieved": achieved, "frac": achieved / peak, "kernel_ms": kernel_ms, "algorithmic_bytes": int(alg_bytes),
            "kernel": "bmx::expand_kernel" if W["dense"] else "bmx::scan_kernel", "step_gpu_ms": step_gpu_ms,
            "step_algorithmic_bytes": int(step_bytes), "step_achieved": step_bytes / (step_gpu_ms * 1e-3) / 1e9,
            "step_frac": step_bytes / (step_gpu_ms * 1e-3) / 1e9 / peak}


def instrumented_repeats(scanner, W, pos, stream, reps):
    """The library's CUDA events around the scan kernel alone and around scan + expand, on the launching stream."""
    scanner.set_timing(2)
    scan_ms, whole_ms = [], []
    for _ in range(reps):
        scanner.begin(pos, stream=stream)
        scanner.scan(W["text"], W["lo"], stream=stream)
        c, st = scanner.finish(stream=stream)
        scan_ms.append(st["scan_kernel_ms"])
        whole_ms.append(st["device_ms"])
    return c, st, float(np.mean(scan_ms)), float(np.mean(whole_ms))


def measure_config(bmx, torch, name, dev, local, args, peak):
    """One of the other BASELINE configs on one GPU: K back-to-back scans (device-timed), the kernel's
    roofline, and the oracle's verdict.  Returns the entry of the line's `configs` table."""
    W = build_workload(bmx, torch, name, 1, 0, dev)
    pos = torch.empty(W["cap"], dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    scanner = bmx.Scanner(local)
    scanner.set_pattern(W["pat"], variant=args.variant, stream=stream)
    steps = max(5, min(args.steps, 20 if W["w"]["n"] >= GIB else 200))
    scanner.set_timing(0)
    for _ in range(3):
        scanner.begin(pos, stream=stream)
        scanner.scan(W["text"], W["lo"], stream=stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        scanner.begin(pos, stream=stream)
        scanner.scan(W["text"], W["lo"], stream=stream)
    e1.record()
    torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / steps
    count, st, scan_ms, gpu_ms = instrumented_repeats(scanner, W, pos, stream, 5)
    ok, how, ocount, _ = oracle_verdict(torch, W["text"], W["lo"], W["pat"], count, pos, W["cap"], W["dense"])
    ok = ok and verify_hits(torch, W["text"], W["lo"], W["pat"], pos, count, W["cap"])
    n = W["end"] - W["lo"]
    rf = kernel_roofline(W, count, scan_ms, gpu_ms, peak)
    scanner.close()
    return {"value": n / (ms_step * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": ms_step, "steps": steps, "bytes": int(n),
            "pattern_len": W["m"], "alphabet": W["w"]["alphabet"], "variant": st["variant"], "hits": int(count),
            "oracle_hits": int(ocount), "verified": bool(ok), "verified_by": how,
            "roofline": {"frac": rf["frac"], "achieved": rf["achieved"], "kernel": rf["kernel"], "kernel_ms": rf["kernel_ms"],
                         "algorithmic_bytes": rf["algorithmic_bytes"], "step_frac": rf["step_frac"]}}


def e2e_balanced_leg(bmx, bd, torch, dist, w, pat, plants, total_n, world, rank, local, dev, e2e_cap, e2e_steps, total_hits, old_host):
    """e2e with shards proportional to each rank's host->device rate, measured with all ranks copying at once.
    Returns the e2e record, or None when the rates are within 10 % of each other (nothing to balance)."""
    m = len(pat)
    alpha = bmx.synth.ALPHABETS[w["alphabet"]]
    probe_h = torch.empty(256 << 20, dtype=torch.uint8, pin_memory=True)
    probe_d = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    probe_d.copy_(probe_h, non_blocking=True)
    torch.cuda.synchronize()
    dist.barrier()
    t0, copied = time.perf_counter(), 0
    while time.perf_counter() - t0 < 0.25:          # every rank copies for the same 250 ms: all links busy throughout
        probe_d.copy_(probe_h, non_blocking=True)
        torch.cuda.synchronize()
        copied += probe_h.numel()
    rate = copied / (time.perf_counter() - t0)
    rates = torch.zeros(world, dtype=torch.float64, device=dev)
    rates[rank] = rate
    dist.all_reduce(rates)
    rates = rates.cpu().tolist()
    del probe_h, probe_d
    if max(rates) < 1.10 * min(rates) and not os.environ.get("BMX_BENCH_FORCE_BALANCE"):   # (test knob)
        return None
    # rank r owns the start positions [cut[r], cut[r+1]) of the same global text; cuts are 16-byte aligned
    total_rate, acc, cut = sum(rates), 0.0, [0]
    for r in range(world - 1):
        acc += rates[r]
        cut.append(min(total_n, int(total_n * acc / total_rate) // 16 * 16))
    cut.append(total_n)
    lo2, hi2 = cut[rank], cut[rank + 1]
    end2 = min(total_n, hi2 + m - 1)
    shard = torch.empty(end2 - lo2, dtype=torch.uint8, device=dev)
    bmx.synth.fill_device(shard, lo2, w["seed"], alpha)
    bmx.synth.plant_device(shard, pat, plants[(plants + m > lo2) & (plants < end2)], base=lo2)
    if old_host is not None and old_host.numel() >= end2 - lo2:
        host = old_host[: end2 - lo2]              # the equal-shard buffer is big enough: no second pinned allocation
    else:
        del old_host
        host = torch.empty(end2 - lo2, dtype=torch.uint8, pin_memory=True)
    host.copy_(shard)
    torch.cuda.synchronize()
    del shard
    bmx.search(host, pat, max_positions=e2e_cap, device=local)          # warm-up (buffers grow to the new shard size)
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        c2, p2 = bmx.search(host, pat, max_positions=e2e_cap, device=local)
        tot, _, _ = bd.combine_hits(c2, torch.from_numpy(p2 + lo2).to(dev), group=None, device=dev)
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    if int(tot) != int(total_hits):
        raise RuntimeError(f"balanced shards found {tot} hits, the device-resident run {total_hits}")
    return {"value": total_n / (float(dt.item()) / e2e_steps) / 1e9, "unit": "GB/s", "steps": e2e_steps,
            "h2d_bytes_per_step": int(end2 - lo2) + m + 1024 + 4 * m, "d2h_bytes_per_step": 8 * int(min(c2, e2e_cap)) + 8,
            "api": "bmx_search_ex (host pointers, pinned text)",
            "shards": "proportional to each rank's host->device rate, all ranks copying at once",
            "rank_rates_gbs": [round(x / 1e9, 1) for x in rates], "rank0_shard_bytes": int(cut[1] - cut[0])}


def run_ours(args):
    import torch
    import torch.distributed as dist

    import parallel_implementation_of_string_matching_algorithms_opencl_b200 as bmx
    from parallel_implementation_of_string_matching_algorithms_opencl_b200 import distributed as bd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: there is no CPU path"
    # Placement: with fewer ranks than GPUs the ranks are spread over the box (every (G/N)-th GPU) instead of packed on
    # GPUs 0..N-1: on the 8-GPU boxes of this pool GPUs 0-3 share one ~115 GB/s path to host memory while 4-7 each get
    # their full 55 GB/s (profiles/ingest_topology_r02.txt), so four packed ranks ingest at 29 GB/s each and four
    # spread ranks at 54 GB/s.  The device-resident numbers do not depend on it.  BMX_BENCH_PLACEMENT=packed restores 0..N-1.
    local_rank = local
    ngpu = torch.cuda.device_count()
    placement = "packed"
    if world > 1 and ngpu > world and ngpu % world == 0 and os.environ.get("BMX_BENCH_PLACEMENT", "spread") == "spread" \
            and int(os.environ.get("LOCAL_WORLD_SIZE", world)) == world:
        local = local_rank * (ngpu // world)
        placement = f"spread (every {ngpu // world}th of {ngpu} GPUs)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bd.bind_to_device_numa(local) if not args.no_numa_bind else None   # pinned text + staging threads next to the GPU's PCIe root
    if os.environ.get("NCCL_DEBUG", "VERSION") == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"          # keep NCCL's version banner off stdout (one JSON line only)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    name = args.workload or ("dna_m32_4GiB" if world == 1 else "ascii95_m64_shard")
    W = build_workload(bmx, torch, name, world, rank, dev, args.bytes_per_gpu)
    w, m, total_n, lo, end, pat, plants, text, dense, cap = (W[k] for k in ("w", "m", "total_n", "lo", "end", "pat", "plants", "text", "dense", "cap"))
    peak, peak_src = peaks()

    pos = torch.empty(cap, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    scanner = bmx.Scanner(local)
    scanner.set_pattern(pat, variant=args.variant, stream=stream)

    # N > 1: the exchange step runs inside the library over NVLink peer memory (bmx_exchange_*): behind scan i the
    # post kernel stores {count, list head} into every rank's mailbox, and the collect kernel of step i-1 (sum of
    # counts everywhere, concatenated list on rank 0) is enqueued behind it -- no collective kernel competing for
    # SMs with the persistent scan grid, no host synchronisation inside the loop.  --exchange nccl keeps round 1's
    # torch.distributed all-gather for comparison.
    xchg = None
    exchange_kind = "none"
    if world > 1:
        exchange_kind = args.exchange
        if exchange_kind == "peer":
            try:
                xchg = bd.PeerExchange(dev, head_cap=bd.FAST_GATHER_CAP, tail_cap=(cap if dense else 0))
            except Exception as e:   # no peer access / IPC on this box: say so and use the NCCL exchange
                print(f"[rank {rank}] peer exchange unavailable ({e}); falling back to NCCL", file=sys.stderr, flush=True)
                exchange_kind = "nccl (peer exchange unavailable)"
            flag = torch.tensor([1 if xchg is not None else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if not int(flag.item()):
                xchg = None
                exchange_kind = "nccl (peer exchange unavailable)"
    gathered = [torch.empty(min(cap * world, 1 << 26) if rank == 0 else 1, dtype=torch.int64, device=dev) for _ in range(2)] if xchg else None
    depth = 3 if (world > 1 and xchg is None) else 1
    ring = [(pos if i == 0 else torch.empty(cap, dtype=torch.int64, device=dev),
             torch.zeros(2 + bd.FAST_GATHER_CAP, dtype=torch.int64, device=dev)) for i in range(depth)] if world > 1 and xchg is None else None
    inflight = []
    state = {"i": 0, "last": None, "host": [0.0, 0.0, 0.0]}

    def step():
        if world == 1:
            scanner.begin(pos, stream=stream)
            scanner.scan(text, lo, stream=stream)
            return
        t0 = time.perf_counter()
        i = state["i"]
        state["i"] += 1
        if xchg is not None:
            scanner.begin(pos, stream=stream)
            scanner.scan(text, lo, stream=stream)
            t1 = time.perf_counter()
            xchg.post(scanner, stream)
            t2 = time.perf_counter()
            if i > 0:
                state["seq"] = xchg.collect(gathered[(i - 1) & 1] if rank == 0 else None, stream)
            t3 = time.perf_counter()
            state["host"] = [a + b for a, b in zip(state["host"], (t1 - t0, t2 - t1, t3 - t2))]
            return
        if len(inflight) == depth:
            state["last"] = inflight.pop(0).finish()
        t1 = time.perf_counter()
        p_i, packed_i = ring[i % depth]
        scanner.begin(p_i, stream=stream)
        scanner.scan(text, lo, stream=stream)
        scanner.export_result(packed_i, stream=stream)
        t2 = time.perf_counter()
        inflight.append(bd.combine_hits_start(None, p_i, group=None, device=dev, packed=packed_i))
        t3 = time.perf_counter()
        state["host"] = [a + b for a, b in zip(state["host"], (t1 - t0, t2 - t1, t3 - t2))]

    def drain():
        if xchg is not None:
            if state["i"] > 0:
                state["seq"] = xchg.collect(gathered[(state["i"] - 1) & 1] if rank == 0 else None, stream)
                state["i"] = 0       # the next step() starts a fresh post/collect pairing
            return
        while inflight:
            state["last"] = inflight.pop(0).finish()

    for _ in range(args.warmup):
        step()
    drain()
    count, stats = scanner.finish(stream=stream)
    ok = verify_hits(torch, text, lo, pat, pos, count, cap)

    # Everything that costs host time (NVML set-up: milliseconds, and it contends across processes) happens BEFORE the
    # barrier: round 1's "3.4 ms one-off at 8 GPUs" was start skew between the ranks -- each rank initialised NVML
    # between the barrier and its first event, and the ranks that started early waited in their first exchange
    # for the one that started last (profiles/r02_n8_timeline.txt).
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    scanner.set_timing(0)          # no event records between the kernels of the headline loop (they cost ~10 us/step)
    state["host"] = [0.0, 0.0, 0.0]
    with ClockSampler(local) as clk:
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
        clk.arm()
        t_host0 = time.perf_counter()
        e0.record()
        for _ in range(args.steps):
            step()
        drain()
        e1.record()
        t_host1 = time.perf_counter()
        torch.cuda.synchronize()
        t_host2 = time.perf_counter()
        if world > 1:
            dist.barrier()
    count, stats = scanner.finish(stream=stream)
    ms_total = ms_local = e0.elapsed_time(e1)
    total_hits = count
    counts_all, gathered_len, gathered_list = [count], min(count, cap), (pos[: min(count, cap)] if world == 1 else None)
    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
        if xchg is not None:
            total_hits, counts_all, gathered_len = xchg.wait(state["seq"])
            if rank == 0:
                gathered_list = gathered[(args.steps - 1) & 1][:gathered_len]
        elif state["last"] is not None:
            total_hits, counts_all, gathered_list = state["last"]
            gathered_len = 0 if gathered_list is None else int(gathered_list.numel())
        ok = ok and total_hits == sum(counts_all) and counts_all[rank] == count
    if args.dump_outputs and rank == 0:      # before the instrumented repeats below reuse the position buffer
        dump_outputs(torch, args.dump_outputs, total_hits, gathered_list)
    ms_step = ms_total / args.steps
    value = total_n / (ms_step * 1e-3) / 1e9

    # instrumented repeat of the same steps (local scan only), right after the timed loop
    torch.cuda.synchronize()
    kreps = max(3, min(args.steps, 20))
    _c, stats, stats_scan_ms, step_gpu_ms = instrumented_repeats(scanner, W, pos, stream, kreps)
    rf = kernel_roofline(W, count, stats_scan_ms, step_gpu_ms, peak)
    traffic = None
    for tf in (ROOT / "profiles" / "r02_traffic.json", ROOT / "profiles" / "r01_traffic.json"):
        if tf.exists() and traffic is None:
            rec = json.loads(tf.read_text()).get(name)
            if rec and not args.bytes_per_gpu:
                traffic = rec["dram_read_bytes"] + rec["dram_write_bytes"]

    # ---- the oracle's verdict (outside every timed region): every rank's local result against the reference's
    # serial code on the same shard; rank 0's gathered list against the rank-ordered concatenation of the oracle lists
    verified_by = "not run (--no-verify)"
    oracle_hits = None
    host_text = None
    if not (args.no_verify and args.no_e2e):     # one pinned host copy of the shard serves the oracle and the e2e leg
        host_text = torch.empty(end - lo, dtype=torch.uint8, pin_memory=True)
        host_text.copy_(text)
        torch.cuda.synchronize()
    if not args.no_verify:
        ok_local, verified_by, ocount, opos = oracle_verdict(torch, text, lo, pat, count, pos, cap, dense, host=host_text.numpy())
        ok = ok and ok_local
        oracle_hits = ocount
        if world > 1:
            lists = [None] * world
            dist.all_gather_object(lists, (int(ocount), None if opos is None else (opos + lo)))
            oracle_hits = sum(c for c, _ in lists)
            ok = ok and oracle_hits == total_hits
            if rank == 0 and not dense and gathered_list is not None:
                want = np.concatenate([p for _, p in lists])
                ok = ok and np.array_equal(gathered_list.cpu().numpy(), want[:gathered_len]) and gathered_len == min(want.size, gathered[0].numel() if xchg else want.size)
            flag = torch.tensor([1 if ok else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            ok = bool(flag.item())
            verified_by += f"; every rank's shard + the gathered list on rank 0 ({world} ranks)"

    # ---- e2e: host-pointer C-ABI call, H2D + scan + D2H inside the timed region (pinned text; pageable text
    # -- the reference's own calling pattern, std::string -> malloc copy, BoyreMoore.cpp:77-90 -- at N = 1)
    e2e = e2e_pageable = None
    host_sample = None
    if not args.no_e2e:
        e2e_cap = min(cap, 1 << 24)
        e2e_steps = max(2, min(args.steps, args.e2e_steps))

        def e2e_run(src, label):
            bmx.search(src, pat, max_positions=e2e_cap, device=local)     # warm-up (allocations)
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                c2, p2 = bmx.search(src, pat, max_positions=e2e_cap, device=local)
                if world > 1:
                    bd.combine_hits(c2, torch.from_numpy(p2 + lo).to(dev), group=None, device=dev)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if world > 1:
                t = torch.tensor([dt], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            return c2, {"value": total_n / (dt / e2e_steps) / 1e9, "unit": "GB/s", "steps": e2e_steps,
                        "h2d_bytes_per_step": int(end - lo) + len(pat) + 1024 + 4 * len(pat),
                        "d2h_bytes_per_step": 8 * int(min(c2, e2e_cap)) + 8, "api": f"bmx_search_ex (host pointers, {label} text)"}

        c2, e2e = e2e_run(host_text, "pinned")
        ok = ok and c2 == count
        host_sample = host_text
        # N > 1: the GPUs of a box need not ingest at the same rate (8-GPU boxes of this pool: 23 GB/s per GPU on one half,
        # 35 on the other when all eight copy at once, profiles/ingest_topology_r02.txt), and equal shards finish with
        # the slowest link.  Second leg: the SAME global text cut in proportion to each rank's measured host->device rate.
        if world > 1 and not args.no_balance:
            try:
                old_host, host_text, host_sample = host_text, None, None     # the leg reuses or replaces the pinned buffer
                bal = e2e_balanced_leg(bmx, bd, torch, dist, w, pat, plants, total_n, world, rank, local, dev, e2e_cap, e2e_steps, total_hits, old_host)
                del old_host
            except Exception as exc:   # noqa: BLE001 -- the equal-shard figure stands
                print(f"[rank {rank}] balanced e2e leg failed: {exc!r}", file=sys.stderr, flush=True)
                bal = None
            flag = torch.tensor([1 if bal is not None else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) and bal["value"] > e2e["value"]:
                bal["equal_shards"] = {"value": e2e["value"], "unit": "GB/s"}
                e2e = bal
        if world == 1 and not args.no_pageable:
            pageable = host_text.numpy().copy()
            c3, e2e_pageable = e2e_run(pageable, "pageable")
            ok = ok and c3 == count
            del pageable

    # ---- cpu_baseline: the reference's own serial code on a bounded sample (rank 0, N = 1)
    cpu = None
    if world == 1 and not args.no_cpu and rank == 0:
        cpu = cpu_baseline(host_sample if host_sample is not None else text.cpu(), pat, threads=1,
                           sample_bytes=args.cpu_sample_bytes)
        if cpu["sample_bytes"] == end - lo:
            ok = ok and cpu["hits"] == count       # the baseline leg scanned the whole text: same count

    if os.environ.get("BENCH_DEBUG"):
        n_steps = max(args.steps, 1)
        print(f"[rank {rank}] numa={numa} exchange={exchange_kind} gpu_ms(local events)={ms_local:.3f} max-over-ranks={ms_total:.3f} "
              f"step_gpu_ms={step_gpu_ms:.4f} host enqueue of {n_steps} steps={(t_host1 - t_host0) * 1e3:.3f} ms "
              f"(scan {state['host'][0] / n_steps * 1e6:.1f} us, post {state['host'][1] / n_steps * 1e6:.1f} us, collect {state['host'][2] / n_steps * 1e6:.1f} us per step) "
              f"sync after enqueue={(t_host2 - t_host1) * 1e3:.3f} ms", file=sys.stderr, flush=True)

    # ---- the other BASELINE configs (N = 1): same protocol, one entry each in `configs`
    configs = None
    if world == 1 and not args.no_configs and not args.workload:
        del text, pos
        W["text"] = None
        torch.cuda.empty_cache()
        configs = {name: {"value": value, "unit": "GB/s", "ms_per_step": ms_step, "steps": args.steps, "bytes": int(end - lo),
                          "pattern_len": m, "alphabet": w["alphabet"], "variant": stats["variant"], "hits": int(total_hits),
                          "oracle_hits": oracle_hits, "verified": bool(ok), "verified_by": verified_by,
                          "roofline": {k: rf[k] for k in ("frac", "achieved", "kernel", "kernel_ms", "algorithmic_bytes", "step_frac")}}}
        for other in ("ascii95_m16_64MiB", "bytes256_m4_4GiB", "bytes256_m16_4GiB", "bytes256_m128_4GiB", "aaa_1GiB", "ascii95_m64_shard"):
            configs[other] = measure_config(bmx, torch, other, dev, local, args, peak)
            torch.cuda.empty_cache()
        for c in configs.values():
            c["baseline_config"] = True
        for other in EXTRA_CONFIGS:      # mid-density and short-pattern cases (see WORKLOADS)
            configs[other] = measure_config(bmx, torch, other, dev, local, args, peak)
            configs[other]["baseline_config"] = False
            torch.cuda.empty_cache()

    if rank == 0:
        launches_per_step = 2 if world == 1 else (4 if xchg is not None else 3)
        line = {
            "metric": "text GB/s scanned (device-timed)", "value": value, "unit": "GB/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": name, "bytes_per_gpu": int(w["n"]), "total_bytes": int(total_n), "pattern_len": m,
                       "alphabet": w["alphabet"], "plants": int(len(plants)), "hits": int(total_hits), "oracle_hits": oracle_hits,
                       "variant": stats["variant"], "tile_bytes": stats["tile_bytes"], "stages": stats["stages"],
                       "grid": stats["grid"], "l2": "inputs larger than L2 (no flush needed)" if w["n"] > (256 << 20) else "input fits L2: flushless, see DESIGN.md",
                       "verified": bool(ok), "verified_by": verified_by, "exchange": exchange_kind, "placement": placement, "gpu_index": local,
                       "numa_node": numa, "parallelism": f"shard{world}" if world > 1 else "single"},
            "roofline": {"bound": "hbm", "achieved": rf["achieved"], "peak": peak, "unit": "GB/s", "frac": rf["frac"],
                         "traffic": traffic, "peak_source": peak_src, "kernel_ms": rf["kernel_ms"],
                         "algorithmic_bytes": rf["algorithmic_bytes"], "kernel": rf["kernel"],
                         "kernel_timing": f"CUDA events recorded by libbmx around the kernel, mean of {kreps} instrumented repeats right after the timed loop",
                         "step_gpu_ms": rf["step_gpu_ms"], "step_algorithmic_bytes": rf["step_algorithmic_bytes"],
                         "step_achieved": rf["step_achieved"], "step_frac": rf["step_frac"]},
            "e2e": e2e, "e2e_pageable": e2e_pageable, "gpu_launches": int(args.steps) * launches_per_step,
            "clocks": clk.summary(), "cpu_baseline": cpu, "configs": configs,
        }
        emit(line)
    scanner.close()
    if world > 1:
        dist.barrier()
        if xchg is not None:
            xchg.close()
        dist.destroy_process_group()


def cpu_baseline(host_text, pat, threads: int, sample_bytes: int):
    """Times oracle/_ref/libref_bm.so (the reference's own code) -- or the oracle port when the
    reference build is absent -- on a bounded prefix of the text."""
    arr = host_text.numpy() if hasattr(host_text, "numpy") else host_text
    n = int(min(arr.size, sample_bytes))
    cnt = ctypes.c_uint64()
    ref_so = ROOT / "oracle" / "_ref" / "libref_bm.so"
    legal7 = len(pat) <= 99 and max(pat) < 0x80 and int(arr[: min(n, 1 << 24)].max()) < 0x80
    if ref_so.exists() and legal7:
        lib, kind = ctypes.CDLL(str(ref_so)), "reference"
        fn = lib.ref_bm_search_windowed
    else:
        so = ROOT / "oracle" / "liboracle.so"
        if not so.exists():
            import subprocess
            subprocess.run(["bash", str(ROOT / "oracle" / "build_oracle.sh")], check=True, capture_output=True)
        lib, kind = ctypes.CDLL(str(so)), "port"
        fn = lib.oracle_search_mt
    t0 = time.perf_counter()
    rc = fn(ctypes.c_void_p(arr.ctypes.data), ctypes.c_int64(n), ctypes.c_char_p(pat), ctypes.c_int32(len(pat)),
            None, ctypes.c_int64(0), ctypes.byref(cnt), ctypes.c_int32(threads))
    dt = time.perf_counter() - t0
    assert rc == 0, rc
    return {"value": n / dt / 1e9, "unit": "GB/s", "cores": threads if threads > 0 else os.cpu_count(), "kind": kind,
            "sample": f"first {n} bytes of the workload text, {cnt.value} hits, {dt:.2f} s", "host_cores_total": os.cpu_count(),
            "hits": int(cnt.value), "sample_bytes": n}


def run_reference(args):
    """The reference's own CPU implementation of the path on all host threads (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    import parallel_implementation_of_string_matching_algorithms_opencl_b200.synth as synth

    name = args.workload or ("dna_m32_4GiB" if world == 1 else "ascii95_m64_shard")
    w = dict(WORKLOADS[name])
    alpha = synth.ALPHABETS[w["alphabet"]]
    total_n = w["n"] * world
    n = int(min(w["n"], args.cpu_sample_bytes))          # bounded sample: a prefix of the text
    so = ROOT / "oracle" / "liboracle.so"
    if not so.exists():
        import subprocess
        subprocess.run(["bash", str(ROOT / "oracle" / "build_oracle.sh")], check=True, capture_output=True)
    orc = ctypes.CDLL(str(so))
    text = np.empty(n, dtype=np.uint8)
    chunk = 64 << 20

    def fill(lo):
        ln = min(chunk, n - lo)
        orc.oracle_synth_fill(ctypes.c_void_p(text.ctypes.data + lo), ctypes.c_int64(lo), ctypes.c_int64(ln),
                              ctypes.c_uint64(w["seed"]), ctypes.c_char_p(alpha), len(alpha))
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
        list(ex.map(fill, range(0, n, chunk)))

    class _B:  # minimal stand-in so make_pattern/plant_list can be shared
        pass
    b = _B()
    b.synth = synth
    pat = make_pattern(b, w, total_n)
    plants = plant_list(b, w, total_n, world)
    synth.plant_host(text, pat, plants[plants < n])

    threads = os.cpu_count() or 1
    res = cpu_baseline(text, pat, threads=-1, sample_bytes=n)       # warm-up, also sizes the sample
    rate = res["value"] * 1e9
    budget_s = 120.0                                                  # the whole K-step run stays within minutes
    if n / rate * args.steps > budget_s:
        n = max(64 << 20, int(rate * budget_s / args.steps) // (64 << 20) * (64 << 20))
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = cpu_baseline(text, pat, threads=-1, sample_bytes=n)
    dt = (time.perf_counter() - t0) / args.steps
    value = n / dt / 1e9
    res["value"] = value
    res["cores"] = threads
    emit({
        "impl": "reference", "metric": "text GB/s scanned (device-timed)", "value": value, "unit": "GB/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": name, "bytes_per_gpu": int(w["n"]), "total_bytes": int(total_n), "pattern_len": w["m"],
                   "alphabet": w["alphabet"], "sample_bytes": n,
                   "note": "reference serial BM (its own kernel1.cl + BoyreMoore.cpp tables) run window-parallel on all host threads"},
        "cpu_baseline": res, "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)   # 200 back-to-back 4 GiB scans run into sw_power_cap on these boxes (-1.8 %)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--variant", default="auto")
    ap.add_argument("--bytes-per-gpu", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="skip the oracle comparison (outside the timed regions)")
    ap.add_argument("--no-configs", action="store_true", help="N = 1: skip the other BASELINE configs")
    ap.add_argument("--no-pageable", action="store_true", help="N = 1: skip the pageable-text e2e leg")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--no-balance", action="store_true", help="N > 1: skip the e2e leg with shards proportional to the ranks' ingest rates")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"], help="N > 1: exchange step over peer memory (library) or NCCL all-gather")
    ap.add_argument("--cpu-sample-bytes", type=int, default=4 * GIB)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the count and positions of the last timed step to DIR as .npy (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    # stdout carries exactly ONE JSON line: libraries that chat on fd 1 (NCCL's version banner)
    # are sent to stderr for the duration of the run
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
