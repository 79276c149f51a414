"""Multi-GPU plumbing for the sharded scene preparation (one process per GPU, torch.distributed).

Sharding: every rank owns a contiguous entity range (all views), culls and sorts it with the single-GPU path; the sorted
(key, payload) runs are then exchanged by key range and merged so that the result equals a single sort over all entities,
ties broken by global entity order (ranks hold contiguous ranges in rank order, the merge breaks ties by (rank, payload)).

The exchange itself lives in libgarden_sceneprep.so (csrc/exchange.cu, csrc/merge.cu: NCCL loaded by the library, no host
synchronisation, key-range all-to-all + merge-path tree) — `PipelinedRunMerger` below only carries the NCCL unique id over
torch.distributed and forwards to gsp_exchange_*.

`plan_gather`, `pack_block`, `plan_from_blocks`, `sample_run`, `common_splitters`, `split_bounds` and `merge_reference` are
pure numpy statements of what the device kernels compute (layouts, splitters, expected merges); the CPU tests check them,
including world_size-2 gloo runs of the count exchange, the one-block all-gather and the all-to-all.
"""
from __future__ import annotations

import numpy as np


def plan_gather(counts: np.ndarray):
    """counts: [ranks, lists] list lengths. Returns (offsets [ranks, lists], rank_stride, out_offsets [lists], totals [lists]).

    Every rank packs its lists back to back; rank r's block starts at r * rank_stride in the gathered buffer;
    the merged list l is at out_offsets[l] (sized for the whole list, a rank only fills its slice)."""
    counts = np.asarray(counts, dtype=np.int64)
    offsets = np.zeros_like(counts)
    offsets[:, 1:] = np.cumsum(counts, axis=1)[:, :-1]
    rank_stride = int(max(1, counts.sum(axis=1).max()))
    totals = counts.sum(axis=0)
    out_offsets = np.zeros(counts.shape[1], dtype=np.int64)
    out_offsets[1:] = np.cumsum(totals)[:-1]
    return offsets.astype(np.uint32), rank_stride, out_offsets.astype(np.uint32), totals.astype(np.uint32)


# ---- the packed exchange block (garden_b200/csrc/merge.cu: kExportPacked / kMergePlan), stated in numpy -----------------
EX_HEADER_WORDS, EX_HEADER_FIXED, EX_MAGIC = 256, 8, 0x47535031


def pack_block(list_keys, list_payloads, capacity: int) -> np.ndarray:
    """What kExportPacked writes for one rank: header {magic, lists, total, capacity, overflow, 0, 0, 0, count[lists]} |
    keys[capacity] | payloads[capacity]. An overflowing rank (total > capacity) carries zero counts and no elements."""
    lists = len(list_keys)
    assert lists <= EX_HEADER_WORDS - EX_HEADER_FIXED
    block = np.zeros(EX_HEADER_WORDS + 2 * capacity, dtype=np.uint32)
    counts = np.array([len(k) for k in list_keys], dtype=np.int64)
    total = int(counts.sum())
    overflow = total > capacity
    block[0:5] = [EX_MAGIC, lists, total, capacity, 1 if overflow else 0]
    if not overflow:
        block[EX_HEADER_FIXED:EX_HEADER_FIXED + lists] = counts
        if total:
            block[EX_HEADER_WORDS:EX_HEADER_WORDS + total] = np.concatenate(list_keys)
            block[EX_HEADER_WORDS + capacity:EX_HEADER_WORDS + capacity + total] = np.concatenate(list_payloads)
    return block


def plan_from_blocks(gathered: np.ndarray, ranks: int, lists: int, capacity: int, out_capacity: int):
    """What kMergePlan derives from the gathered blocks: (offsets [ranks, lists], counts [ranks, lists], out_offsets [lists],
    flags [8]) with flags = {error bits (1 overflow, 2 bad header, 4 merged lists exceed out_capacity), merged total,
    largest per-rank total, 0...}. With a non-zero error word every count is zero (nothing may be merged)."""
    words = EX_HEADER_WORDS + 2 * capacity
    hdr = np.asarray(gathered, dtype=np.uint32).reshape(ranks, words)[:, :EX_HEADER_WORDS]
    error = 0
    for r in range(ranks):
        if hdr[r, 0] != EX_MAGIC or hdr[r, 1] != lists:
            error |= 2
        if hdr[r, 4]:
            error |= 1
    counts = np.zeros((ranks, lists), dtype=np.int64) if error else hdr[:, EX_HEADER_FIXED:EX_HEADER_FIXED + lists].astype(np.int64)
    offsets = np.zeros_like(counts)
    offsets[:, 1:] = np.cumsum(counts, axis=1)[:, :-1]
    totals = counts.sum(axis=0)
    out_offsets = np.zeros(lists, dtype=np.int64)
    out_offsets[1:] = np.cumsum(totals)[:-1]
    merged = int(totals.sum())
    if merged > out_capacity:
        error |= 4
        counts = np.zeros_like(counts)
    flags = np.zeros(8, dtype=np.int64)
    flags[0], flags[1], flags[2] = error, merged, int(hdr[:, 2].max())
    return offsets, counts, out_offsets, flags


# ---- the all-to-all protocol (garden_b200/csrc/merge.cu: kSampleRuns / kSplitRuns / kPackByDestination), stated in numpy ------
EX_SAMPLES = 64


def sample_run(keys: np.ndarray) -> np.ndarray:
    """What kSampleRuns writes for one sorted run: EX_SAMPLES keys at positions (2k + 1) * n / (2 * EX_SAMPLES), then n."""
    n = len(keys)
    out = np.full(EX_SAMPLES + 1, 0xFFFFFFFF, dtype=np.uint32)
    if n:
        pos = ((2 * np.arange(EX_SAMPLES, dtype=np.uint64) + 1) * np.uint64(n)) // np.uint64(2 * EX_SAMPLES)
        out[:EX_SAMPLES] = np.asarray(keys, dtype=np.uint32)[pos.astype(np.int64)]
    out[EX_SAMPLES] = n
    return out


def common_splitters(samples: np.ndarray) -> np.ndarray:
    """samples: [ranks, EX_SAMPLES + 1] of ONE list (every rank holds the same array after the all-gather).
    Splitter j (j = 1 .. ranks-1) = the smallest key x whose weighted rank W(x) = sum_r n_r * #(samples of r <= x) reaches
    ceil(j / ranks * sum_r n_r * EX_SAMPLES) — integer arithmetic, identical on every rank (kSplitRuns)."""
    samples = np.asarray(samples, dtype=np.uint64)
    ranks = samples.shape[0]
    weights = samples[:, EX_SAMPLES]
    total = int(weights.sum()) * EX_SAMPLES
    out = np.full(max(ranks - 1, 0), 0xFFFFFFFF, dtype=np.uint32)
    if total == 0:
        return out
    for j in range(1, ranks):
        target = (total * j + ranks - 1) // ranks
        lo, hi = 0, 0xFFFFFFFF
        while lo < hi:
            mid = lo + ((hi - lo) >> 1)
            w = sum(int(weights[r]) * int(np.searchsorted(samples[r, :EX_SAMPLES], mid, side="right")) for r in range(ranks)
                    if weights[r])
            if w >= target:
                hi = mid
            else:
                lo = mid + 1
        out[j - 1] = lo
    return out


def split_bounds(keys: np.ndarray, splitters: np.ndarray) -> np.ndarray:
    """[ranks + 1] cut positions of one sorted run: destination d gets keys[b[d]:b[d+1]]; a key equal to a splitter starts
    the next range."""
    keys = np.asarray(keys, dtype=np.uint32)
    inner = np.searchsorted(keys, np.asarray(splitters, dtype=np.uint32), side="left")
    return np.concatenate([[0], np.maximum.accumulate(inner), [len(keys)]]).astype(np.int64)


def merge_reference(runs_keys, runs_payloads, my_rank: int | None = None):
    """numpy statement of the merge for ONE list: runs_* are per-rank arrays (sorted by key, ties by payload).
    Returns (keys, payloads, ranks) of the full merged list, or of rank `my_rank`'s key-range slice plus its start."""
    ranks = len(runs_keys)
    keys = np.concatenate(runs_keys) if ranks else np.zeros(0, np.uint32)
    pays = np.concatenate(runs_payloads) if ranks else np.zeros(0, np.uint32)
    src = np.concatenate([np.full(len(k), r, np.uint8) for r, k in enumerate(runs_keys)]) if ranks else np.zeros(0, np.uint8)
    order = np.lexsort((pays, src, keys))  # key, then rank, then payload
    keys, pays, src = keys[order], pays[order], src[order]
    if my_rank is None:
        return keys, pays, src
    run0 = runs_keys[int(np.argmax([len(k) for k in runs_keys]))]  # longest run, lowest rank on ties
    n0 = len(run0)
    lo_key = run0[my_rank * n0 // ranks] if (my_rank > 0 and n0) else None
    hi_key = run0[(my_rank + 1) * n0 // ranks] if (my_rank + 1 < ranks and n0) else None
    lo = int(np.searchsorted(keys, lo_key, side="left")) if lo_key is not None else 0
    hi = int(np.searchsorted(keys, hi_key, side="left")) if hi_key is not None else len(keys)
    hi = max(hi, lo)
    return keys[lo:hi], pays[lo:hi], src[lo:hi], lo


def merge_path_cut(a: np.ndarray, b: np.ndarray, diag: int) -> int:
    """How many of the first `diag` outputs of merge(a, b) come from a, a winning ties — the binary search kTreePartition's
    warps run (csrc/merge.cu: warpMergePath, 32 probes per round there)."""
    lo, hi = max(0, diag - len(b)), min(diag, len(a))
    while lo < hi:
        mid = (lo + hi) // 2
        if a[mid] <= b[diag - 1 - mid]:
            lo = mid + 1
        else:
            hi = mid
    return lo


def merge_tree_reference(runs_keys, runs_payloads, tile: int = 2048):
    """numpy statement of the pairwise merge tree (kTreePartition + kMergeTree) for ONE list: the runs are merged two by
    two in rank order, level by level, every merge cut into tiles of `tile` outputs by merge-path diagonals and each tile
    merged on its own (a wins ties). Returns (keys, payloads, ranks) — equal to merge_reference(...) of the same runs."""
    groups = [(np.asarray(k, np.uint32), np.asarray(p, np.uint32), np.full(len(k), r, np.uint8))
              for r, (k, p) in enumerate(zip(runs_keys, runs_payloads))]
    if not groups:
        return np.zeros(0, np.uint32), np.zeros(0, np.uint32), np.zeros(0, np.uint8)
    while len(groups) > 1:
        merged = []
        for g in range(0, len(groups), 2):
            if g + 1 == len(groups):
                merged.append(groups[g])  # (an odd group is copied through: a merge with an empty partner)
                continue
            (ka, pa, ra), (kb, pb, rb) = groups[g], groups[g + 1]
            n = len(ka) + len(kb)
            out_k, out_p, out_r = np.empty(n, np.uint32), np.empty(n, np.uint32), np.empty(n, np.uint8)
            for d0 in range(0, n, tile):
                d1 = min(d0 + tile, n)
                i0, i1 = merge_path_cut(ka, kb, d0), merge_path_cut(ka, kb, d1)
                j0, j1 = d0 - i0, d1 - i1
                ta, tb = ka[i0:i1], kb[j0:j1]
                # inside the tile: an element of a goes after the b's that are smaller, an element of b after the a's <= it
                pos_a = np.arange(len(ta)) + np.searchsorted(tb, ta, side="left")
                pos_b = np.arange(len(tb)) + np.searchsorted(ta, tb, side="right")
                out_k[d0 + pos_a], out_p[d0 + pos_a], out_r[d0 + pos_a] = ta, pa[i0:i1], ra[i0:i1]
                out_k[d0 + pos_b], out_p[d0 + pos_b], out_r[d0 + pos_b] = tb, pb[j0:j1], rb[j0:j1]
            merged.append((out_k, out_p, out_r))
        groups = merged
    return groups[0]


def exchange_counts(counts: np.ndarray, group=None) -> np.ndarray:
    """All-gather of the per-list lengths. Works with any backend (tensors live where the backend needs them)."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    backend = dist.get_backend(group)
    device = torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu")
    mine = torch.as_tensor(np.asarray(counts, dtype=np.int64), device=device)
    out = torch.empty(world * mine.numel(), dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(out, mine, group=group)
    return out.cpu().numpy().reshape(world, mine.numel())


class PipelinedRunMerger:
    """The exchange of libgarden_sceneprep.so (csrc/exchange.cu: NCCL inside the library, no Python in the data path), driven
    one rank per process. This class only (a) carries the NCCL unique id from rank 0 to the others over torch.distributed
    and (b) forwards to gsp_exchange_*:

        frame()   gsp_run_async + gsp_exchange_async   — no host synchronisation; frame k's exchange (the library's exchange
                  stream) overlaps frame k+1's culling; buffer sets are double-buffered inside the library
        poll()    gsp_exchange_poll: flags of finished frames; a frame whose runs overflowed the fixed-capacity blocks was
                  not merged: grow() and repeat it
        finish()  gsp_exchange_finish: the compute stream waits for the exchanges, the host for their flags

    Protocol: GSP_EXCHANGE=alltoall (default: sample-based common splitters, every rank receives only its key range) or
    allgather (every rank receives every run)."""

    HEAD_ROOM = 1.25

    def __init__(self, sp, capacity: int | None = None, overlap: bool = True):
        import ctypes as C
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.sp, self.C = torch, dist, sp, C
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        self.overlap = overlap
        lib = sp.lib
        ident = torch.zeros(128, dtype=torch.uint8)
        if self.rank == 0:
            buf = (C.c_uint8 * 128)()
            if lib.gsp_comm_unique_id(buf) != 0:
                raise RuntimeError("gsp_comm_unique_id failed (is libnccl.so.2 loadable?)")
            ident = torch.tensor(list(buf), dtype=torch.uint8)
        backend = dist.get_backend()
        if backend == "nccl":
            ident = ident.cuda()
        dist.broadcast(ident, src=0)
        raw = bytes(ident.cpu().tolist())
        sp._check(lib.gsp_comm_init(sp.h, raw, self.world, self.rank))
        if capacity is None:
            cap = C.c_uint32()
            sp._check(lib.gsp_exchange_autosize(sp.h, C.byref(cap)))
            self.capacity = cap.value
        else:
            sp.run()
            sp._check(lib.gsp_exchange_configure(sp.h, int(capacity)))
            self.capacity = int(capacity)
        self.lists = sp.list_count()
        info = [C.c_uint32() for _ in range(4)]
        sp._check(lib.gsp_comm_info(sp.h, *[C.byref(i) for i in info]))
        self.all_to_all = bool(info[3].value)
        # kernels of this library per frame on top of the single-GPU frame (NCCL's own kernels are not counted):
        # alltoall: kSampleRuns, kSplitRuns, kPackByDestination, kMergePlan, kMergeBounds, kSliceStarts + (kTreePartition,
        # kMergeTree) per merge level; allgather: kExportPacked, kMergePlan, kMergeBounds + the same per level
        levels = max(1, int(np.ceil(np.log2(max(self.world, 2)))))
        self.launches_per_frame = (6 if self.all_to_all else 3) + 2 * levels
        self.timing = None
        self.frame_index = 0

    def grow(self, needed: int):
        """Re-sizes the blocks for `needed` elements (collective: every rank must call it with the same value)."""
        self.finish(check=False)
        self.capacity = int(needed * self.HEAD_ROOM) + 4096
        self.sp._check(self.sp.lib.gsp_exchange_configure(self.sp.h, self.capacity))

    def frame(self):
        sp = self.sp
        sp.run_async()
        if self.timing is not None:
            sp.lib.gsp_exchange_set_timing(sp.h, 1)
        sp._check(sp.lib.gsp_exchange_async(sp.h))
        if self.timing is not None:
            ms = (self.C.c_float * 3)()
            sp._check(sp.lib.gsp_exchange_times(sp.h, ms))  # (synchronises: only used by the serialised latency loop)
            self.timing.append(tuple(ms))
        self.frame_index += 1
        if not self.overlap:
            self.finish()

    def _flags(self, wait: bool, finish: bool):
        C, sp = self.C, self.sp
        bits, needed = C.c_uint32(), C.c_uint32()
        if finish:
            sp._check(sp.lib.gsp_exchange_finish(sp.h, C.byref(bits), C.byref(needed)))
        else:
            sp._check(sp.lib.gsp_exchange_poll(sp.h, 1 if wait else 0, C.byref(bits), C.byref(needed)))
        return [(self.frame_index - 1, bits.value, needed.value)] if bits.value else []

    def poll(self, wait: bool = False):
        """[(frame, error bits, needed capacity)] of the finished frames that failed (empty: everything seen so far is clean)."""
        return self._flags(wait, False)

    def finish(self, check: bool = True):
        failed = self._flags(True, True)
        if check and failed:
            raise RuntimeError(f"exchange overflow in frames {failed}: call grow() and repeat them")
        return failed

    def timing_summary(self):
        if not self.timing:
            return None
        n = len(self.timing)
        return {"export_or_sampling_ms": sum(t[0] for t in self.timing) / n, "collectives_ms": sum(t[1] for t in self.timing) / n,
                "merge_ms": sum(t[2] for t in self.timing) / n, "frames": n,
                "protocol": "alltoall" if self.all_to_all else "allgather"}

    def bytes_received(self) -> int:
        return int(self.sp.lib.gsp_exchange_bytes_received(self.sp.h))

    def last_result(self):
        """This rank's merged slices of the most recent frame on the host (for tests): synchronises."""
        C, sp = self.C, self.sp
        slices = []
        for l in range(self.lists):
            k, p, r = C.c_void_p(), C.c_void_p(), C.c_void_p()
            start, count = C.c_uint32(), C.c_uint32()
            sp._check(sp.lib.gsp_get_merged_device(sp.h, l, C.byref(k), C.byref(p), C.byref(r), C.byref(start), C.byref(count)))
            n = count.value
            keys, pays, ranks = np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.zeros(n, np.uint8)
            if n:
                sp._check(sp.lib.gsp_copy_to_host(sp.h, k, keys.ctypes.data, n * 4))
                sp._check(sp.lib.gsp_copy_to_host(sp.h, p, pays.ctypes.data, n * 4))
                sp._check(sp.lib.gsp_copy_to_host(sp.h, r, ranks.ctypes.data, n))
            slices.append((start.value, keys, pays, ranks))
        return {"slices": slices, "bytes_received": self.bytes_received()}
