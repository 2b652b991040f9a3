"""Multi-GPU sharding of the scan: one process per GPU, torch.distributed for the plumbing.

The reference has no multi-device path (one OpenCL device, BoyreMoore.cpp:217-219); its only
partitioning is the host's word split into P ranges WITHOUT overlap, which loses matches that
straddle a seam (BoyreMoore.cpp:119-141, SURVEY.md A.5).  Here rank r owns the match START
positions [lo_r, hi_r) and reads (m-1) bytes of halo behind hi_r, so every occurrence is reported
exactly once by the rank that owns its start, with its global offset (pos_base = lo_r).

Exchange step (the only exchange on the path), two implementations:

  PeerExchange   (default on GPUs) -- the library's own exchange (bmx_exchange_*, csrc/bmx_exchange.cu): every
                 rank stores {count, head of its list} straight into its peers' mailboxes over NVLink (cudaIpc
                 mappings between the processes), a collect kernel sums the counts and concatenates the lists on
                 rank 0.  Two tiny kernels per step on the scan's own stream, no host synchronisation, no
                 collective kernel waiting for SMs behind the persistent scan grid.  torch.distributed is used
                 once, at set-up, to pass the 64-byte IPC handles around.
  combine_hits   ONE all_gather (NCCL on GPUs, gloo in the CPU tests) carrying each rank's count and (the head
                 of) its position list; every rank sums the counts, rank 0 concatenates the lists in rank order,
                 which is already globally ascending.  Longer lists send their tail to rank 0 point-to-point.
"""
from __future__ import annotations

from typing import Callable, Optional

SHARD_ALIGN = 16  # shard starts are 16-byte aligned so each rank's TMA tiles stay aligned


def shard_bounds(n_total: int, world: int, rank: int) -> tuple[int, int]:
    """Start positions [lo, hi) owned by `rank` (contiguous, disjoint, covering [0, n_total))."""
    per = -(-n_total // world)
    per = -(-per // SHARD_ALIGN) * SHARD_ALIGN
    lo = min(n_total, rank * per)
    hi = min(n_total, (rank + 1) * per)
    return lo, hi


def shard_read_range(n_total: int, m: int, lo: int, hi: int) -> tuple[int, int]:
    """Bytes [lo, end) a rank must hold: its own range plus the (m-1)-byte halo."""
    return lo, min(n_total, hi + max(m - 1, 0))


def bind_to_device_numa(device_index: int):
    """Pins the calling process (and the threads it starts later: the library's staging threads) to the CPUs
    of the NUMA node the GPU's PCIe root hangs off, so that pinned host buffers (first touch) and the
    pageable->pinned staging copies stay on the GPU's side of the socket interconnect.  Returns the node, or
    None when the topology is not visible (then nothing is changed)."""
    import os

    try:
        import torch
        p = torch.cuda.get_device_properties(device_index)
        bus = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


class PeerExchange:
    """One process per GPU: this rank's bmx_exchange wired to its peers through cudaIpc handles that travel
    in one all_gather at set-up.  Every phase ends with an agreement so that a rank that cannot take part
    (no peer access, IPC refused) fails the set-up on ALL ranks instead of leaving the others hanging."""

    def __init__(self, device, group=None, dst: int = 0, head_cap: int = 4096, tail_cap: int = 0, depth: int = 4):
        import torch
        import torch.distributed as dist

        from .host import Exchange

        world, rank = dist.get_world_size(group), dist.get_rank(group)

        def agree(ok: bool, what: str, err):
            flag = torch.tensor([1 if ok else 0], device=device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
            if not int(flag.item()):
                raise RuntimeError(f"peer exchange: {what} failed on some rank" + (f" (here: {err})" if err else ""))

        self.x, err = None, None
        try:
            self.x = Exchange(device.index, rank, world, dst, head_cap, tail_cap, depth)
            handle = self.x.handle()
        except Exception as e:   # noqa: BLE001 -- reported through agree()
            err, handle = e, bytes(Exchange.HANDLE_BYTES)
        agree(err is None, "creating the mailbox", err)
        mine = torch.frombuffer(bytearray(handle), dtype=torch.uint8).to(device)
        everyone = torch.empty(world * Exchange.HANDLE_BYTES, dtype=torch.uint8, device=device)
        dist.all_gather_into_tensor(everyone, mine, group=group)
        try:
            self.x.connect(everyone.cpu().numpy().tobytes())
        except Exception as e:   # noqa: BLE001
            err = e
        agree(err is None, "mapping the peers' mailboxes", err)
        self.rank, self.world, self.dst = rank, world, dst

    def post(self, scanner, stream=0) -> int:
        return self.x.post(scanner, stream)

    def collect(self, out=None, stream=0) -> int:
        return self.x.collect(out, stream)

    def wait(self, seq: int):
        return self.x.wait(seq)

    def close(self):
        if self.x is not None:
            self.x.close()
            self.x = None


class PendingExchange:
    """Collectives of one exchange step, enqueued but not yet awaited (see combine_hits_start)."""

    def __init__(self, works, everyone, width, fast_cap, positions_local, group, dst, device):
        self.works, self.everyone = works, everyone
        self.width, self.fast_cap, self.positions_local = width, fast_cap, positions_local
        self.group, self.dst, self.device = group, dst, device

    def finish(self):
        """Waits for the collectives (the step's single host sync) and assembles the list on dst.
        Returns (total_count, per_rank_counts, positions_on_dst_or_None).

        The list on dst is a prefix of the global ascending list, as the library exchange delivers it: whole
        lists in rank order up to and including the first rank that holds fewer positions than its count.
        Every rank knows every (count, held) pair from the gathered header, so every rank computes the same
        cut; ranks behind it send no tail and dst posts no receive for them.

        On CUDA everything here runs on a side stream that depends only on the collectives, so a
        caller that has already queued later scans on its compute stream is not held up by them."""
        import contextlib

        import torch
        import torch.distributed as dist

        cuda = self.device.type == "cuda"
        side = _side_stream(self.device) if cuda else None
        with (torch.cuda.stream(side) if cuda else contextlib.nullcontext()):
            for w in self.works:
                w.wait()
            world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
            table = self.everyone.view(world, self.width)
            header_dev = table[:, :2].reshape(-1)
            if cuda:
                header = torch.empty(header_dev.numel(), dtype=torch.int64, pin_memory=True)
                header.copy_(header_dev, non_blocking=True)
                side.synchronize()                                     # the single host sync
            else:
                header = header_dev
            header = header.tolist()
            counts_host = [int(header[2 * r]) for r in range(world)]
            held_host = [int(header[2 * r + 1]) for r in range(world)]
            total_host = sum(counts_host)                              # every rank holds every count
            fast_cap, pos = self.fast_cap, self.positions_local
            take, complete = [], True                                  # the same cut on every rank
            for c, h in zip(counts_host, held_host):
                take.append(min(c, h) if complete else 0)
                complete = complete and h >= c

            gathered = None
            if rank == self.dst:
                heads = [table[r, 2: 2 + min(take[r], fast_cap)] for r in range(world)]
                if all(t <= fast_cap for t in take):
                    gathered = torch.cat(heads) if heads else torch.empty(0, dtype=torch.int64, device=self.device)
                else:
                    gathered = torch.empty(sum(take), dtype=torch.int64, device=self.device)
                    off, reqs = 0, []
                    for r in range(world):
                        k = min(take[r], fast_cap)
                        if k:
                            gathered[off: off + k] = heads[r]
                        rest = take[r] - k
                        if rest > 0:
                            if r == self.dst:
                                gathered[off + k: off + k + rest] = pos[k: k + rest]
                            else:
                                reqs.append(dist.irecv(gathered[off + k: off + k + rest], src=r, group=self.group))
                        off += take[r]
                    for q in reqs:
                        q.wait()
            elif take[rank] > fast_cap:
                dist.send(pos[fast_cap:take[rank]].contiguous(), dst=self.dst, group=self.group)
        if cuda:
            torch.cuda.current_stream(self.device).wait_stream(side)   # later users of `gathered` are ordered after it
        return total_host, counts_host, gathered


_SIDE_STREAMS = {}


def _side_stream(device):
    import torch

    key = (device.type, device.index)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
    return _SIDE_STREAMS[key]


FAST_GATHER_CAP = 4096  # positions per rank that ride along with the count exchange


def combine_hits_start(count_local, positions_local, *, group=None, device=None, dst: int = 0,
                       fast_cap: int = FAST_GATHER_CAP, packed=None) -> PendingExchange:
    """Enqueues the exchange step and returns without waiting.

    positions_local: 1-D int64 tensor of this rank's GLOBAL positions (ascending), on `device`
    (it may hold fewer than count_local entries when the caller capped its output).
    packed: optional int64[2 + fast_cap] tensor on `device` that already holds (or, stream-ordered,
    will hold) {count, positions written, head of the list} -- Scanner.export_result() -- in which
    case count_local is ignored, positions_local is the whole output buffer, and nothing here waits
    for the scan: the collectives are enqueued behind it.

    One all-gather carries every rank's [count, list length, first fast_cap positions] (the global
    count is the sum of the gathered counts: no separate all-reduce).  PendingExchange.finish() awaits it
    with a single host synchronisation; lists longer than fast_cap (dense texts) send their remainder to
    `dst` point-to-point.  Rank-order concatenation on `dst` is globally ascending: nothing is sorted.
    The list on `dst` is a prefix of the global list, the same one the library exchange returns: it stops
    behind the first rank whose list holds fewer positions than its count.
    """
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    device = device if device is not None else positions_local.device
    width = 2 + fast_cap
    if packed is None:
        held_local = 0 if positions_local is None else int(positions_local.numel())
        mine = torch.empty(width, dtype=torch.int64, device=device)
        mine[:2] = torch.tensor([int(count_local), held_local], dtype=torch.int64)
        k_local = min(held_local, fast_cap)
        if k_local:
            mine[2: 2 + k_local] = positions_local[:k_local]
    else:
        assert packed.numel() == width and packed.dtype == torch.int64
        mine = packed

    works = []
    everyone = torch.empty(world * width, dtype=torch.int64, device=device)
    try:
        works.append(dist.all_gather_into_tensor(everyone, mine, group=group, async_op=True))
    except (RuntimeError, NotImplementedError):
        _all_gather_list(everyone, mine, group)
    return PendingExchange(works, everyone, width, fast_cap, positions_local, group, dst, device)


def combine_hits(count_local, positions_local, **kw):
    """Exchange step, blocking: combine_hits_start(...).finish()."""
    return combine_hits_start(count_local, positions_local, **kw).finish()


def _all_gather_list(out, mine, group):
    import torch
    import torch.distributed as dist

    parts = [torch.empty_like(mine) for _ in range(dist.get_world_size(group))]
    dist.all_gather(parts, mine, group=group)
    out.copy_(torch.cat(parts))


def sharded_search(shard_text, lo: int, pattern: bytes, *, max_positions: int, group=None, dst: int = 0,
                   variant="auto", local_scan: Optional[Callable] = None, fast_cap: int = FAST_GATHER_CAP):
    """Scan this rank's shard and run the exchange step.

    shard_text holds the bytes [lo, end) of the global text (own range + halo, see
    shard_read_range).  Returns (total_count, per_rank_counts, positions_on_dst_or_None,
    local_stats).  The positions on dst are a prefix of the global ascending list: whole shard lists in
    rank order, ending behind the first rank that found more than max_positions.
    `local_scan(shard_text, pattern, pos_base, max_positions)` ->
    (count, positions_tensor, stats) defaults to the CUDA scan; the CPU tests inject a checker.
    """
    if local_scan is None:
        from .host import search_device

        def local_scan(text, pat, pos_base, cap):
            return search_device(text, pat, max_positions=cap, pos_base=pos_base, variant=variant)

    count, pos, stats = local_scan(shard_text, pattern, lo, max_positions)
    total, counts, gathered = combine_hits(count, pos, group=group, device=shard_text.device, dst=dst, fast_cap=fast_cap)
    return total, counts, gathered, stats
