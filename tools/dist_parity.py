#!/usr/bin/env python
"""Real multi-GPU parity check of the sharded path (run under torchrun, one rank per GPU, NCCL):

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tools/dist_parity.py

One scene is cut into world_size contiguous entity ranges (at chain boundaries); every rank prepares its range and the
library's exchange (garden_b200.dist.PipelinedRunMerger: NCCL inside the library, protocol chosen by GSP_EXCHANGE) merges
the sorted runs, three frames in flight. Every rank then checks its merged key-range slice bit for bit against the numpy
statement of the merge (dist.merge_reference) applied to the runs of ALL ranks (collected over the object channel) and that
the slices tile every list with no gap or overlap; then the same after overflow -> grow -> repeat. Prints one JSON line on
rank 0. The emulated-rank version of the same check is tests/test_gpu_merge.py.
"""
from __future__ import annotations

import json
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from garden_b200 import scenes, views as V  # noqa: E402
from garden_b200.dist import PipelinedRunMerger, merge_reference, plan_gather  # noqa: E402


def main():
    import torch
    import torch.distributed as dist
    from garden_b200.binding import ScenePrep

    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    chains, depth = 40000, 4
    n = chains * (depth + 1)
    whole = scenes.make_scene(n, depth, 5, (-150, -10, -150, 150, 10, 150))
    whole.camera_pos = np.array([2.0, 1.0, -3.0], np.float32)
    views, _ = V.camera_and_cascades(0.3, -0.1, 1.2, 16 / 9, 0.01, 100.0, (0.05, 0.1, 0.25, 1.0))
    per = (chains // world) * (depth + 1)
    starts = [r * per for r in range(world)] + [n]
    a, b = starts[rank], starts[rank + 1]
    shard = scenes.SceneDesc(whole.position[a:b], whole.rotation[a:b], whole.scale[a:b],
                             np.where(whole.parent[a:b] >= 0, whole.parent[a:b] - a, -1).astype(np.int32), whole.tflags[a:b],
                             [scenes.PoolDesc(whole.pools[0].render_type, np.arange(b - a, dtype=np.uint32),
                                              whole.pools[0].aabb[a:b])], None, whole.camera_pos)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sp = ScenePrep(local)
    sp.set_stream(stream.cuda_stream)
    t, pools = scenes.build_aos(shard)
    sp.set_transforms(t, t.dtype.itemsize, t.size)
    sp.set_pool_count(len(pools))
    for k, m in enumerate(pools):
        sp.set_mesh_pool(k, shard.pools[k].render_type, m, m.dtype.itemsize, m.size)
    sp.set_views(views, shard.camera_pos)
    sp.run()

    # this rank's own runs, for the object-channel cross-check
    counts = sp.list_counts().astype(np.int64)
    total = int(counts.sum())
    k = torch.empty(max(total, 1), dtype=torch.int32, device="cuda")
    p = torch.empty(max(total, 1), dtype=torch.int32, device="cuda")
    sp.export_runs(k.data_ptr(), p.data_ptr(), max(total, 1))
    sp.sync()
    torch.cuda.synchronize()
    mine = (counts, k[:total].cpu().numpy().view(np.uint32), p[:total].cpu().numpy().view(np.uint32))
    everyone = [None] * world
    dist.all_gather_object(everyone, mine)
    all_counts = np.stack([c for c, _, _ in everyone])
    offsets, _, _, totals = plan_gather(all_counts)
    lists = counts.size
    # ---- the exchange INSIDE the library (csrc/exchange.cu: NCCL behind the C ABI, no host synchronisation): three frames in
    # flight, every slice against the numpy merge of ALL ranks' runs, then the overflow path ----
    full = []
    for l in range(lists):
        runs_k = [everyone[r][1][offsets[r, l]: offsets[r, l] + all_counts[r, l]] for r in range(world)]
        runs_p = [everyone[r][2][offsets[r, l]: offsets[r, l] + all_counts[r, l]] for r in range(world)]
        full.append(merge_reference(runs_k, runs_p))

    def check_slices(result, what):
        for l in range(lists):
            start, gk, gp, gr = result["slices"][l]
            fk, fp, fr = full[l]
            sl = slice(start, start + gk.size)
            assert start + gk.size <= fk.size, f"rank {rank} list {l} ({what}): slice [{start}, {start + gk.size}) outside the list"
            assert np.array_equal(gk, fk[sl]) and np.array_equal(gp, fp[sl]) and np.array_equal(gr, fr[sl]), \
                f"rank {rank} list {l} ({what}): merged slice differs from the merge of all runs"
        spans = [None] * world
        dist.all_gather_object(spans, [(s[0], int(s[1].size)) for s in result["slices"]])
        for l in range(lists):
            pos = 0
            for r in range(world):
                assert spans[r][l][0] == pos, f"list {l} ({what}): rank {r} slice starts at {spans[r][l][0]}, expected {pos}"
                pos += spans[r][l][1]
            assert pos == int(totals[l]), f"list {l} ({what}): slices cover {pos} of {int(totals[l])}"
        return spans

    pm = PipelinedRunMerger(sp)
    for _ in range(3):
        pm.frame()
        assert pm.poll() == []
    pm.finish()
    spans_lib = check_slices(pm.last_result(), "in-library exchange")
    protocol = "alltoall" if pm.all_to_all else "allgather"
    small = max(int(all_counts.sum(axis=1).max()) // (3 * (world if pm.all_to_all else 1)), 1)
    pm.finish()
    sp.run()
    sp._check(sp.lib.gsp_exchange_configure(sp.h, small))
    pm.capacity = small
    pm.frame()
    failed = pm.finish(check=False)
    assert failed and failed[0][1] & 1 and failed[0][2] > small, failed
    need = torch.tensor([failed[0][2]], dtype=torch.int64, device="cuda")
    dist.all_reduce(need, op=dist.ReduceOp.MAX)
    pm.grow(int(need.item()))
    pm.frame()
    assert pm.finish(check=False) == []
    check_slices(pm.last_result(), "after overflow -> grow -> repeat")
    if rank == 0:
        print(json.dumps({"dist_parity": "ok", "world": world, "entities": n, "lists": int(lists),
                          "merged_total": int(totals.sum()),
                          "in_library_exchange": f"ok ({protocol}; 3 frames in flight, overflow -> grow -> repeat)",
                          "bytes_received_per_rank": pm.bytes_received(),
                          "slice_lengths_list0": [s[0][1] for s in spans_lib]}), flush=True)
    sp.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
