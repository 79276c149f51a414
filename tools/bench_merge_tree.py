#!/usr/bin/env python
"""Single-GPU timing of the exchange's merge (gsp_merge_gathered_packed_tree) with the ranks emulated: `ranks` blocks of
sorted runs laid out as the collective leaves them, merged as rank `me`. Runs are `ranks` times longer than a real
all-to-all sub-block, so that the slice this rank merges has the size it has in a real frame (--slice elements).

  python tools/bench_merge_tree.py --ranks 8 --slice 4400000 [--lists 5] [--reps 50] [--check]
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    import torch
    from garden_b200.binding import load_library
    ap = argparse.ArgumentParser()
    ap.add_argument("--ranks", type=int, default=8)
    ap.add_argument("--slice", type=int, default=4_400_000)
    ap.add_argument("--lists", type=int, default=5)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--check", action="store_true")
    a = ap.parse_args()
    lib = load_library()
    ranks, lists = a.ranks, a.lists
    g = torch.Generator(device="cuda").manual_seed(7)
    # list lengths like a C4 frame: the camera list holds half, the cascades share the rest
    share = np.array([0.5] + [0.5 / max(lists - 1, 1)] * (lists - 1))[:lists]
    share /= share.sum()
    per_run = [int(a.slice * s) for s in share]  # elements of list l in EVERY run (=> slice ~ per_run[l] per list)
    cap = sum(per_run) + 64
    words = lib.gsp_exchange_block_words(cap)
    gathered = torch.zeros(words * ranks, dtype=torch.int32, device="cuda")
    for r in range(ranks):
        hdr = np.zeros(256, np.uint32)
        hdr[:5] = (0x47535031, lists, sum(per_run), cap, 0)
        hdr[8:8 + lists] = per_run
        gathered[r * words:r * words + 256] = torch.from_numpy(hdr.view(np.int32)).cuda()
        at = 0
        for l in range(lists):
            n = per_run[l]
            k = torch.randint(0, 1 << 30, (n,), generator=g, device="cuda", dtype=torch.int32).sort().values
            gathered[r * words + 256 + at:r * words + 256 + at + n] = k
            gathered[r * words + 256 + cap + at:r * words + 256 + cap + at + n] = torch.arange(n, device="cuda", dtype=torch.int32)
            at += n
    total = sum(per_run) * ranks
    plan = torch.zeros(lib.gsp_merge_plan_words(ranks, lists), dtype=torch.int32, device="cuda")
    sinfo = torch.zeros(lists * 2, dtype=torch.int32, device="cuda")
    out_k = torch.zeros(total, dtype=torch.int32, device="cuda"); out_p = torch.zeros_like(out_k)
    out_r = torch.zeros(total, dtype=torch.uint8, device="cuda")
    scratch = torch.zeros(int(lib.gsp_merge_tree_scratch_words(total)), dtype=torch.int32, device="cuda")
    me = ranks // 2

    def once():
        rc = lib.gsp_merge_gathered_packed_tree(0, ranks, me, lists, cap, gathered.data_ptr(), plan.data_ptr(), sinfo.data_ptr(),
                                                out_k.data_ptr(), out_p.data_ptr(), out_r.data_ptr(), total, scratch.data_ptr())
        assert rc == 0
    torch.cuda.set_stream(torch.cuda.default_stream())
    for _ in range(5):
        once()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.reps):
        once()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.reps
    info = sinfo.cpu().numpy().reshape(lists, 2)
    merged = int(info[:, 1].sum())
    res = {"ranks": ranks, "lists": lists, "merged_elements": merged, "ms": ms,
           "GBps_per_level_equiv": merged * 18 / ms / 1e6}
    if a.check:
        offs = np.concatenate([[0], np.cumsum(np.array(per_run) * ranks)[:-1]])
        ok = True
        kk, rr = out_k.cpu().numpy(), out_r.cpu().numpy()
        for l in range(lists):
            seg = kk[offs[l]:offs[l] + info[l, 1]]
            ok &= bool(np.all(seg[1:] >= seg[:-1]))
            same = seg[1:] == seg[:-1]
            rs = rr[offs[l]:offs[l] + info[l, 1]]
            ok &= bool(np.all(rs[1:][same] >= rs[:-1][same]))
        res["sorted_and_stable"] = ok
    print(json.dumps(res))


if __name__ == "__main__":
    main()
