"""Multi-GPU `match_list_parallel` (src/matcher/parallel.rs:18-89) — ctypes callers of the C ABI.

The path itself lives in the library (frizbee_b200/csrc/parallel.cu): a communicator (`frz_comm`), one clone of the
matcher per GPU, the haystack list sharded by contiguous index range (shard g holds indices [offset_g, offset_g + n_g)),
each GPU's locally ordered run kept in HBM, ONE ncclAllGather of the runs, the k-way merge (src/k_merge.rs:90-131) on
every GPU, every GPU copying its slice of the merged list to the host buffer.  This module only wraps the entry points:

  Comm.local(n_gpus)                       single process driving n GPUs (what a Rust caller does)
  Comm.from_torch_distributed(device)      one rank per process (torchrun); torch.distributed only ships the 128-byte id
  comm.match_list_parallel(matcher, shards)            frz_match_list_parallel
  comm.match_list_parallel_rank(matcher, shard, off)   frz_match_list_parallel_rank

The numpy helpers at the bottom (shard_bounds, merge_runs_host, all_gather_runs, match_list_parallel_host) are the
host-side SPECIFICATION of the shard/merge logic; the world-size-2 gloo tests (tests/test_parallel_gloo.py) run them on
CPU with the oracle as the run producer.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import MATCH_DTYPE, Corpus, FrizbeeError, Matcher, _arrow_offsets, _check, lib
from .types import SortStrategy

UNIQUE_ID_BYTES = 128


def _bind(L):
    if getattr(L, "_frz_parallel_bound", False):
        return L
    vp, u64, u32 = C.c_void_p, C.c_uint64, C.c_uint32
    L.frz_comm_create_local.argtypes = [C.c_int, vp, C.POINTER(vp)]
    L.frz_comm_unique_id.argtypes = [vp]
    L.frz_comm_create_rank.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
    L.frz_comm_destroy.argtypes = [vp]
    L.frz_comm_destroy.restype = None
    L.frz_comm_world.argtypes = [vp]
    L.frz_comm_rank.argtypes = [vp]
    L.frz_comm_device.argtypes = [vp, C.c_int]
    L.frz_comm_host_alloc.argtypes = [vp, u64, C.POINTER(vp)]
    L.frz_comm_host_free.argtypes = [vp, vp]
    L.frz_comm_barrier.argtypes = [vp]
    L.frz_comm_exchange_mode.argtypes = [vp]
    L.frz_comm_exchange_mode.restype = C.c_int
    L.frz_corpus_create_sharded.argtypes = [vp, vp, C.c_int, u64, vp, C.POINTER(vp)]
    L.frz_match_list_parallel.argtypes = [vp, C.POINTER(vp), C.c_int, vp, vp, u64, C.POINTER(u64)]
    L.frz_match_list_parallel_rank.argtypes = [vp, vp, u32, vp, vp, u64, C.POINTER(u64), C.POINTER(vp)]
    L.frz_match_list_parallel_rank_host.argtypes = [vp, vp, vp, C.c_int, u64, u32, vp, vp, u64, C.POINTER(u64)]
    L.frz_comm_last_timings.argtypes = [vp, C.c_int, C.POINTER(C.c_float), C.POINTER(vp)]
    L.frz_matcher_clone.argtypes = [vp, C.POINTER(vp)]
    L._frz_parallel_bound = True
    return L


def plib():
    return _bind(lib())


class Comm:
    """`frz_comm`: the GPUs one match_list_parallel call runs on."""

    def __init__(self, handle, world: int, rank: int, local_form: bool):
        self._h, self.world, self.rank, self.local_form = handle, world, rank, local_form

    @classmethod
    def local(cls, n_gpus: int, devices: Optional[Sequence[int]] = None) -> "Comm":
        h = C.c_void_p()
        arr = (C.c_int * n_gpus)(*devices) if devices is not None else None
        _check(plib().frz_comm_create_local(n_gpus, arr, C.byref(h)))
        return cls(h, n_gpus, 0, True)

    @staticmethod
    def unique_id() -> bytes:
        buf = (C.c_uint8 * UNIQUE_ID_BYTES)()
        _check(plib().frz_comm_unique_id(buf))
        return bytes(buf)

    @classmethod
    def from_rank(cls, unique_id: bytes, world: int, rank: int, device: int) -> "Comm":
        h = C.c_void_p()
        buf = (C.c_uint8 * UNIQUE_ID_BYTES).from_buffer_copy(unique_id)
        _check(plib().frz_comm_create_rank(buf, world, rank, device, C.byref(h)))
        return cls(h, world, rank, False)

    @classmethod
    def from_torch_distributed(cls, device: int, group=None) -> "Comm":
        """One rank per process: rank 0 draws the NCCL unique id, torch.distributed broadcasts its 128 bytes (the only
        thing torch.distributed does for the data path), every rank joins."""
        import torch
        import torch.distributed as dist
        if not dist.is_initialized():
            return cls.from_rank(cls.unique_id(), 1, 0, device)
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        on_gpu = dist.get_backend(group) == "nccl"
        t = torch.zeros(UNIQUE_ID_BYTES, dtype=torch.uint8, device=torch.device("cuda", device) if on_gpu else "cpu")
        if rank == 0:
            t.copy_(torch.frombuffer(bytearray(cls.unique_id()), dtype=torch.uint8))
        dist.broadcast(t, 0, group=group)
        return cls.from_rank(bytes(t.cpu().numpy().tobytes()), world, rank, device)

    # ---- shared pinned host memory ----
    def host_alloc_matches(self, n: int) -> np.ndarray:
        """A MATCH_DTYPE array in host memory every rank's GPU can write (multi-process: one shared segment; collective)."""
        p = C.c_void_p()
        n = max(int(n), 1)
        _check(plib().frz_comm_host_alloc(self._h, n * MATCH_DTYPE.itemsize, C.byref(p)))
        buf = (C.c_uint8 * (n * MATCH_DTYPE.itemsize)).from_address(p.value)   # memory owned by the communicator
        return np.frombuffer(buf, dtype=MATCH_DTYPE)

    def host_free(self, arr: np.ndarray):
        _check(plib().frz_comm_host_free(self._h, arr.ctypes.data))

    def barrier(self):
        _check(plib().frz_comm_barrier(self._h))

    def exchange_mode(self) -> int:
        """How host-out calls move the matches: 2 = P2P placement, 0 = all-gather."""
        return int(plib().frz_comm_exchange_mode(self._h))

    def p2p_active(self) -> bool:
        return self.exchange_mode() >= 2

    def device(self, local_index: int = 0) -> int:
        return plib().frz_comm_device(self._h, local_index)

    # ---- sharding (local form) ----
    def shard_arrow(self, data: np.ndarray, offsets: np.ndarray) -> List[Corpus]:
        data = np.ascontiguousarray(data, dtype=np.uint8)
        offsets, width = _arrow_offsets(offsets)
        n = len(offsets) - 1
        hs = (C.c_void_p * self.world)()
        _check(plib().frz_corpus_create_sharded(data.ctypes.data if data.size else None, offsets.ctypes.data, width, n, self._h, hs))
        bounds = shard_bounds(n, self.world)
        return [Corpus(C.c_void_p(hs[g]), hi - lo) for g, (lo, hi) in enumerate(bounds)]

    # ---- match_list_parallel ----
    def match_list_parallel(self, matcher: Matcher, shards: Sequence[Corpus], out: Optional[np.ndarray] = None) -> np.ndarray:
        """Local form (frz_match_list_parallel): shards[g] on the communicator's g-th GPU.  Returns the ordered matches."""
        total = sum(len(s) for s in shards)
        if out is None:
            out = np.empty(max(total, 1), dtype=MATCH_DTYPE)
        hs = (C.c_void_p * len(shards))(*[s._h for s in shards])
        n = C.c_uint64()
        _check(plib().frz_match_list_parallel(matcher._h, hs, len(shards), self._h, out.ctypes.data, len(out), C.byref(n)))
        return out[: n.value]

    def match_list_parallel_rank(self, matcher: Matcher, shard: Corpus, index_offset: int, out: Optional[np.ndarray] = None,
                                 want_device: Optional[bool] = None) -> Tuple[int, int]:
        """Multi-process form (frz_match_list_parallel_rank), collective.  `out`: the SHARED host array from
        host_alloc_matches (every rank passes its mapping) or None for a device-only result.  `want_device` (default: only
        when `out` is None) also asks for this rank's device copy of the WHOLE merged list — that forces the all-gather form;
        host-only calls use the P2P placement when peer memory is mapped.  Returns (total matches, device pointer of the merged list or 0)."""
        if want_device is None:
            want_device = out is None
        n = C.c_uint64()
        d = C.c_void_p()
        _check(plib().frz_match_list_parallel_rank(matcher._h, shard._h, index_offset, self._h,
                                                   out.ctypes.data if out is not None else None,
                                                   len(out) if out is not None else 0, C.byref(n),
                                                   C.byref(d) if want_device else None))
        return n.value, d.value or 0

    def match_list_parallel_rank_host(self, matcher: Matcher, data: np.ndarray, offsets: np.ndarray, index_offset: int,
                                      out: np.ndarray) -> int:
        """End to end on one rank: this rank's shard arrives as HOST Arrow buffers (streamed H2D + pack), then the parallel
        match; the merged list lands in the shared host array.  Collective."""
        if offsets.dtype.itemsize == 4 and offsets.flags.c_contiguous:
            width = 4
        else:
            offsets, width = _arrow_offsets(offsets)
        n = C.c_uint64()
        _check(plib().frz_match_list_parallel_rank_host(matcher._h, data.ctypes.data if data.size else None, offsets.ctypes.data,
                                                        width, len(offsets) - 1, index_offset, self._h, out.ctypes.data, len(out),
                                                        C.byref(n)))
        return n.value

    def last_timings(self, local_index: int = 0) -> dict:
        """Device timings of the last parallel call on one local rank + the per-stage timings of the clone that ran it."""
        ms = (C.c_float * 4)()
        clone = C.c_void_p()
        _check(plib().frz_comm_last_timings(self._h, local_index, ms, C.byref(clone)))
        r = {"local_ms": ms[0], "gather_merge_ms": ms[1], "d2h_ms": ms[2], "total_ms": ms[3]}
        if clone.value:
            st = (C.c_float * 4)()
            launches = C.c_uint64()
            _check(lib().frz_matcher_last_timings(clone, st, C.byref(launches)))
            r.update(prefilter_ms=st[0], sw_ms=st[1], sort_ms=st[2], pipeline_ms=st[3], launches=launches.value)
        return r

    def close(self):
        if getattr(self, "_h", None):
            plib().frz_comm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ------------------------------------------------------------------------------------------------------------
# Host-side specification of the shard / merge logic (numpy; used by the gloo tests and as the checker of the device merge)

def shard_bounds(n: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous index ranges, shard g = [g*ceil(n/world), ...) (SURVEY.md §8(e))."""
    per = (n + world - 1) // world if world else 0
    return [(min(g * per, n), min((g + 1) * per, n)) for g in range(world)]


def merge_runs_host(runs: List[np.ndarray], sort: SortStrategy) -> np.ndarray:
    """Reference semantics of k_merge_matches_by_* on host arrays: runs are index-range shards in rank order, each
    ordered per `sort`."""
    if not runs:
        return np.zeros(0, dtype=MATCH_DTYPE)
    cat = np.concatenate(runs[::-1] if sort.is_reversed() else runs)
    if not sort.is_by_score():
        return cat
    order = np.argsort(-cat["score"].astype(np.int64), kind="stable")
    return cat[order]


def placement_host(runs: List[np.ndarray], sort: SortStrategy, bins: int = 1024) -> List[np.ndarray]:
    """Host specification of the P2P placement (csrc/parallel.cu: k_place + the position arithmetic of rank_step): from every
    run's per-score table gt[q][s] (how many elements of run q score higher than s) each rank derives, for ITS run only,
    pos0[s] — the merged position of the first element of its score-s block = everything scoring higher in any run + the
    score-s blocks of the runs that precede it in merge order — and stores element i (score s) at merged position
    pos0[s] + (i - gt[s]), i.e. into slice p = the rank with lo[p] <= position < lo[p + 1], lo[p] = total * p // world.
    Returns the world slices; their concatenation is the k-way merge (tests/test_parallel_gloo.py)."""
    world = len(runs)
    counts = [len(r) for r in runs]
    total = sum(counts)
    lo = [total * p // world for p in range(world + 1)]
    slices = [np.zeros(lo[p + 1] - lo[p], dtype=MATCH_DTYPE) for p in range(world)]
    if total == 0:
        return slices
    by_score = sort.is_by_score()
    nb = bins if by_score else 1
    gt = np.zeros((world, nb), dtype=np.int64)
    if by_score:
        for q, r in enumerate(runs):
            sc = np.minimum(r["score"].astype(np.int64), nb - 1)
            hist = np.bincount(sc, minlength=nb)
            gt[q] = hist[::-1].cumsum()[::-1] - hist          # strictly higher
    ge = np.concatenate([np.asarray(counts, dtype=np.int64)[:, None], gt[:, :-1]], axis=1)   # ge[q][s] = count(score >= s)
    order = list(range(world))[::-1] if sort.is_reversed() else list(range(world))
    for me, r in enumerate(runs):
        pos0 = np.zeros(nb, dtype=np.int64)
        for s in range(nb):
            acc = int(gt[:, s].sum())
            for q in order:
                if q == me:
                    break
                acc += int(ge[q][s] - gt[q][s])
            pos0[s] = acc
        i = np.arange(len(r), dtype=np.int64)
        s_of = np.minimum(r["score"].astype(np.int64), nb - 1) if by_score else np.zeros(len(r), dtype=np.int64)
        x = pos0[s_of] + (i - gt[me][s_of])
        p_of = np.searchsorted(np.asarray(lo[1:], dtype=np.int64), x, side="right")
        for p in range(world):
            sel = p_of == p
            slices[p][x[sel] - lo[p]] = r[sel]
    return slices


def match_list_parallel_placement_gloo(run: np.ndarray, sort: SortStrategy, bins: int = 1024, group=None) -> np.ndarray:
    """The P2P placement protocol of csrc/parallel.cu on torch.distributed (gloo on CPU in the tests), rank-local like on the
    GPUs: (1) every rank publishes its count and its per-score table (all_gather — the shared host block of the device path),
    (2) computes pos0[] for ITS run only, (3) sends every element, tagged with its slice-relative position, to the rank that
    owns that slice of the merged list (all_to_all — the NVLink peer stores of k_place), (4) every rank assembles its slice.
    Returns this rank's slice [total * r // G, total * (r + 1) // G) of the merged list."""
    import torch
    import torch.distributed as dist
    world, me = dist.get_world_size(group), dist.get_rank(group)
    by_score = sort.is_by_score()
    nb = bins if by_score else 1
    mine = np.zeros(nb + 1, dtype=np.int64)            # [count, gt[0..nb)]
    mine[0] = len(run)
    if by_score:
        hist = np.bincount(np.minimum(run["score"].astype(np.int64), nb - 1), minlength=nb)
        mine[1:] = hist[::-1].cumsum()[::-1] - hist
    allt = [torch.zeros(nb + 1, dtype=torch.int64) for _ in range(world)]
    dist.all_gather(allt, torch.from_numpy(mine), group=group)
    tab = np.stack([t.numpy() for t in allt])          # [world][1 + nb]
    counts, gt = tab[:, 0], tab[:, 1:]
    total = int(counts.sum())
    lo = [total * p // world for p in range(world + 1)]
    ge = np.concatenate([counts[:, None], gt[:, :-1]], axis=1)
    order = list(range(world))[::-1] if sort.is_reversed() else list(range(world))
    pos0 = np.zeros(nb, dtype=np.int64)
    for s in range(nb):
        acc = int(gt[:, s].sum())
        for q in order:
            if q == me:
                break
            acc += int(ge[q][s] - gt[q][s])
        pos0[s] = acc
    i = np.arange(len(run), dtype=np.int64)
    s_of = np.minimum(run["score"].astype(np.int64), nb - 1) if by_score else np.zeros(len(run), dtype=np.int64)
    x = pos0[s_of] + (i - gt[me][s_of])
    p_of = np.searchsorted(np.asarray(lo[1:], dtype=np.int64), x, side="right")
    rec = np.ascontiguousarray(run).view(np.int64)
    send = []
    for p in range(world):
        sel = p_of == p
        send.append(torch.from_numpy(np.stack([x[sel] - lo[p], rec[sel]], axis=1).reshape(-1).copy()))   # (position, record) pairs
    sizes = torch.tensor([len(t) for t in send], dtype=torch.int64)
    all_sizes = [torch.zeros(world, dtype=torch.int64) for _ in range(world)]
    dist.all_gather(all_sizes, sizes, group=group)
    recv = [torch.zeros(int(all_sizes[q][me]), dtype=torch.int64) for q in range(world)]
    reqs = [dist.isend(send[p], p, group=group) for p in range(world) if p != me]
    for q in range(world):
        if q == me:
            recv[q] = send[me]
        else:
            dist.recv(recv[q], q, group=group)
    for r in reqs:
        r.wait()
    out = np.zeros(lo[me + 1] - lo[me], dtype=np.int64)
    for t in recv:
        pairs = t.numpy().reshape(-1, 2)
        out[pairs[:, 0]] = pairs[:, 1]
    return out.view(MATCH_DTYPE)


def all_gather_runs(run, count: int, group=None):
    """The collective step on torch tensors (gloo on CPU in the tests): the counts, then ONE all-gather of the runs padded
    to the longest.  `run` is a 1-D int64 tensor of 8-byte match records.  Returns (gathered [world * stride], counts, stride)."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    cnt = torch.tensor([count], dtype=torch.int64, device=run.device)
    counts = torch.zeros(world, dtype=torch.int64, device=run.device)
    dist.all_gather_into_tensor(counts, cnt, group=group)
    counts_h = [int(c) for c in counts.cpu().tolist()]
    stride = max(max(counts_h), 1)
    # a rank whose whole shard is shorter than the longest run (ceil partitioning: the last shard) pads its send buffer
    send = run[:stride].contiguous() if run.numel() >= stride else torch.nn.functional.pad(run, (0, stride - run.numel()))
    gathered = torch.empty(world * stride, dtype=torch.int64, device=run.device)
    dist.all_gather_into_tensor(gathered, send, group=group)
    return gathered, counts_h, stride


def match_list_parallel_host(run: np.ndarray, sort: SortStrategy, group=None) -> np.ndarray:
    """Host/gloo form of the gather + merge (tests; the run producer is injected by the caller)."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(run).view(np.int64).copy())
    gathered, counts, stride = all_gather_runs(t, len(run), group)
    g = gathered.numpy().view(MATCH_DTYPE)
    runs = [g[r * stride: r * stride + counts[r]] for r in range(len(counts))]
    return merge_runs_host(runs, sort)
