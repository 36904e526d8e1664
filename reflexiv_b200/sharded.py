"""Multi-GPU plumbing around the library's sharded calls.

The data path lives in the library (include/reflexiv_cuda.h: rfx_shard_*, csrc/rfx_shard.cu, rfx_shard_graph.cuh): one
context per GPU, every rank's buffers in an arena the other ranks map, kernels reading and writing peer HBM over
NVLink.  What this module adds is the set-up a launcher has to do once: hand every rank the handles of all ranks --
through torch.distributed when there is one process per GPU (`connect`), directly when the ranks are threads of one
process (`LocalRanks`, which is also how a one-GPU box runs the multi-rank path: several ranks share the device).

`sharded_count` is the measured alternative for the counting exchange: records laid out shard-major and moved by one
NCCL all-to-all (the shape of Spark's groupBy shuffle, ReflexivDataFrameCounter.java:198-200) instead of being pulled
out of the peers' slabs by the counting kernel itself.  `exchange_bytes` is backend agnostic (NCCL on GPUs, gloo in
the CPU tests)."""
from __future__ import annotations

from typing import List, Sequence, Tuple


class _DevView:
    """Zero-copy torch view of library-owned device memory (__cuda_array_interface__)."""

    def __init__(self, ptr: int, n_bytes: int):
        self.__cuda_array_interface__ = {"shape": (n_bytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def device_view(torch, ptr: int, n_bytes: int, device):
    if n_bytes == 0:
        return torch.empty(0, dtype=torch.uint8, device=device)
    return torch.as_tensor(_DevView(ptr, n_bytes), device=device)


def shard_of_bin(bin_id: int, n_bins_total: int, n_shards: int) -> int:
    """Bins are shard-major: shard s owns bins [s*B/n, (s+1)*B/n)."""
    return bin_id // (n_bins_total // n_shards)


def choose_total_bins(global_instances: int, n_shards: int, target_per_bin: int = 6144, lo: int = 64, hi: int = 1 << 24) -> int:
    """Same rule as the library's single-process choice (rfx_partition.cu: choose_bin_count; 6144 instances per bin for
    k <= 31, 4096 for k > 31), on the GLOBAL instance count, rounded up to a multiple of the shard count so that every
    rank computes the same number.  With a context at hand prefer ``ctx.choose_bins`` (rfx_choose_bins), which asks
    the library itself."""
    nb = max(lo, min(hi, -(-global_instances // target_per_bin)))
    return -(-nb // n_shards) * n_shards


def exchange_bytes(torch, dist, send, send_sizes: Sequence[int], group=None, alloc=None) -> Tuple[object, List[int]]:
    """All-to-all of variable-size byte slices.  `send` is one uint8 tensor holding the slices for rank 0, 1, ...
    back to back.  Returns (recv tensor, recv sizes).  `alloc(n_bytes)` may supply the receive buffer (e.g. a view of
    memory the library owns, so the received records are counted in place)."""
    world = dist.get_world_size(group)
    assert len(send_sizes) == world and sum(send_sizes) == send.numel()
    s = torch.tensor(list(send_sizes), dtype=torch.int64, device=send.device)
    r = torch.empty(world, dtype=torch.int64, device=send.device)
    dist.all_to_all_single(r, s, group=group)
    recv_sizes = [int(x) for x in r.tolist()]
    recv = alloc(sum(recv_sizes)) if alloc is not None else torch.empty(sum(recv_sizes), dtype=torch.uint8, device=send.device)
    dist.all_to_all_single(recv, send, output_split_sizes=recv_sizes, input_split_sizes=list(send_sizes), group=group)
    return recv, recv_sizes


def gather_varlen(torch, dist, local, group=None):
    """all_gather of tensors of different lengths (same dtype); returns (concatenation in rank order, sizes).
    `local` is 1-D, or [rows, width] with width > 1 (rows vary per rank); sizes are in elements of dim 0.
    One size exchange (a single host read) and one padded all_gather."""
    world = dist.get_world_size(group)
    rows = local.shape[0]
    n = torch.tensor([rows], dtype=torch.int64, device=local.device)
    all_n = torch.empty(world, dtype=torch.int64, device=local.device)
    dist.all_gather_into_tensor(all_n, n, group=group)
    sizes = [int(x) for x in all_n.tolist()]
    mx = max(sizes) if sizes else 0
    shape = (mx,) if local.dim() == 1 else (mx, local.shape[1])
    if rows == mx:
        pad = local.contiguous()
    else:
        pad = torch.zeros(shape, dtype=local.dtype, device=local.device)
        pad[:rows] = local
    flat = torch.empty(world * pad.numel(), dtype=local.dtype, device=local.device)  # flat buffers: gloo accepts nothing else
    dist.all_gather_into_tensor(flat, pad.reshape(-1), group=group)
    out = flat.reshape((world,) + shape)
    if all(sz == mx for sz in sizes):
        return out.reshape((world * mx,) + shape[1:]), sizes
    return torch.cat([out[r, :sizes[r]] for r in range(world)]), sizes


class _Lap:
    """Optional host-side stopwatch (prof dict): laps are cumulative seconds per label, device-synchronised."""

    def __init__(self, torch, device, prof):
        self.torch, self.device, self.prof = torch, device, prof
        if prof is not None:
            import time
            self.time = time
            self.t = time.perf_counter()

    def __call__(self, label):
        if self.prof is None:
            return
        if getattr(self.device, "type", str(self.device)) != "cpu" and self.torch.cuda.is_available():
            self.torch.cuda.synchronize(self.device)
        now = self.time.perf_counter()
        self.prof[label] = self.prof.get(label, 0.0) + now - self.t
        self.t = now


def _sync(torch, device):
    """The library runs on its own stream and its calls block; torch work that produced its inputs must be done."""
    if getattr(device, "type", str(device)) != "cpu" and torch.cuda.is_available():
        torch.cuda.current_stream(device).synchronize()


def sharded_count(ctx, torch, dist, device, n_bins_total: int, group=None, rebin: bool = False, prof=None) -> dict:
    """Counting across the ranks of `group`; on return `ctx` holds this rank's shard of the global table.
    Every sender's slice is already grouped by bin, so its bin offsets travel with it (a second, tiny all-to-all) and
    the owner counts the received buffer in place; `rebin=True` exercises the general path that re-derives the bins."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    lap = _Lap(torch, device, prof)
    ctx.partition(world, n_bins_total)
    lap("count.partition")
    slices = [ctx.shard_records(s) for s in range(world)]
    base = slices[0][0]
    total = sum(n for _, n in slices)
    send = device_view(torch, base, total, device)
    off_ptr, n_off = ctx.shard_bin_offsets(0)
    ctx.begin_shard(rank, world, n_bins_total)
    # receive straight into the context's buffer unless the general (re-binning) path is being exercised
    alloc = None if rebin else (lambda nb: device_view(torch, ctx.rx_buffer(nb), nb, device))
    recv, recv_sizes = exchange_bytes(torch, dist, send, [n for _, n in slices], group, alloc)
    offs_send = device_view(torch, off_ptr, (world * (n_off - 1) + 1) * 8, device).view(torch.int64)
    # shard s needs offsets [s*bps, (s+1)*bps]: bps + 1 values, neighbours share one
    bps = n_off - 1
    idx = (torch.arange(world, device=device).unsqueeze(1) * bps + torch.arange(n_off, device=device).unsqueeze(0)).reshape(-1)
    offs_out = offs_send[idx].contiguous()
    offs_in = torch.empty_like(offs_out)
    dist.all_to_all_single(offs_in, offs_out, group=group)
    _sync(torch, device)
    lap("count.exchange")
    if rebin:
        ctx.load_records_device(recv.data_ptr() if recv.numel() else 0, recv.numel())
    else:
        pos = 0
        for j in range(world):
            ctx.load_segment_device(recv.data_ptr() + pos if recv_sizes[j] else 0, recv_sizes[j], offs_in[j * n_off:(j + 1) * n_off].data_ptr())
            pos += recv_sizes[j]
    del recv
    st = ctx.count()
    lap("count.count")
    return st


_UNEVEN_ALL_GATHER = {}


def _bcast_slices(torch, dist, buf, ranges, group=None):
    """Every rank r owns buf[ranges[r][0]:ranges[r][1]]; after the call every rank holds every slice (in place).
    One all_gather over views of `buf` where the backend takes uneven sizes (NCCL: one grouped launch), else one
    broadcast per rank."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    key = dist.get_backend(group)
    if _UNEVEN_ALL_GATHER.get(key, True):
        try:
            views = [buf[lo:hi] for lo, hi in ranges]
            dist.all_gather(views, views[rank].clone(), group=group)
            _UNEVEN_ALL_GATHER[key] = True
            return
        except (RuntimeError, ValueError, NotImplementedError):
            _UNEVEN_ALL_GATHER[key] = False
    for r in range(world):
        lo, hi = ranges[r]
        if hi > lo:
            dist.broadcast(buf[lo:hi], src=dist.get_global_rank(group, r) if group is not None else r, group=group)


# ---- peer-memory runs: set-up ------------------------------------------------------------------------------------------
def connect(ctx, dist, group=None, arena_bytes: int = 0):
    """One process per GPU: rfx_shard_init on this rank, handles exchanged through `dist` (any backend), peers mapped.
    Afterwards ctx.count_sharded() / ctx.assemble_sharded() are collective calls over the ranks of `group`."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    ctx.shard_init(rank, world, arena_bytes)
    blobs = [None] * world
    dist.all_gather_object(blobs, ctx.shard_export(), group=group)
    ctx.shard_connect(b"".join(blobs), world)


class LocalRanks:
    """Ranks as host threads of one process, one context each (contexts on different GPUs, or sharing one)."""

    def __init__(self, ctxs, arena_bytes: int = 0):
        self.ctxs = list(ctxs)
        world = len(self.ctxs)
        for r, c in enumerate(self.ctxs):
            c.shard_init(r, world, arena_bytes)
        blobs = b"".join(c.shard_export() for c in self.ctxs)
        for c in self.ctxs:
            c.shard_connect(blobs, world)

    def run(self, fn):
        """fn(rank, ctx) on every rank at once (the library calls release the GIL); returns the results in rank order."""
        import threading
        out, err = [None] * len(self.ctxs), [None] * len(self.ctxs)

        def body(r):
            try:
                out[r] = fn(r, self.ctxs[r])
            except BaseException as e:  # noqa: BLE001 -- re-raised below
                err[r] = e

        ts = [threading.Thread(target=body, args=(r,)) for r in range(len(self.ctxs))]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        failed = [(r, e) for r, e in enumerate(err) if e is not None]
        if len(failed) == 1:
            raise failed[0][1]
        if failed:  # a collective call fails on every rank at once; other code in `fn` may fail on some: show every rank's story
            raise RuntimeError("; ".join(f"rank {r}: {e}" for r, e in failed)) from failed[0][1]
        return out
