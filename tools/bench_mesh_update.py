#!/usr/bin/env python
"""Cost of changing mesh components in place on C4 (one GPU): gsp_update_mesh_pool_indexed for 0.1 %, 1 % and 10 % of the
slots, and the frame that follows, against a whole-pool gsp_set_mesh_pool restage. The pool lives in pinned host memory, as
in bench.py's end-to-end arm, and is staged with ready counts so that a getReadyMeshesAsync change can be part of an update.

  python tools/bench_mesh_update.py [--n 16000000] [--reps 5] [--json out.json]

Cases per fraction: `flags` (isEnabled, isVisible and ready-count changes only), `grow` (boxes growing on the listed slots:
rho and the hierarchy spheres widen in place). Times are host clocks around calls that end in a device synchronisation
(gsp_update_mesh_pool* and gsp_run both do), medians over --reps. The run ends by comparing every list of the updated
context with a context freshly staged from the same bytes."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # (reported, not fatal: the numbers still need the card's name beside them)
        out = f"nvidia-smi unavailable: {e}"
    return out


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def all_lists(sp, views):
    out = []
    for v in range(views.size):
        for b in range(sp.unsorted_buffer_count(v)):
            rec, d, i = sp.get_unsorted(v, b)
            out.append((rec.tobytes(), d, i))
        for which in (0, 1):
            rec, d = sp.get_sorted(v, which)
            out.append((rec.tobytes(), d))
    return out


def main():
    from garden_b200 import scenes
    from garden_b200.binding import ScenePrep, pin_host, unpin_host
    import bench
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    info = gpu_info()
    print(f"GPU: {info}", flush=True)

    scene = scenes.config_scene("C4", n=a.n, seed=1234)
    scene.camera_pos = bench.camera_pos()
    views = bench.frame_views("C4")
    t, pools = scenes.build_aos(scene)
    m = pools[0]
    stride, occ = m.dtype.itemsize, m.size
    ready = np.ones(occ, np.uint8)
    for arr in (t, m, ready):
        pin_host(arr)
    rng = np.random.default_rng(5)
    sp = ScenePrep(0)
    sp.set_transforms(t, 80, t.size)
    sp.set_pool_count(1)
    sp.set_mesh_pool(0, scene.pools[0].render_type, m, stride, occ, occ, ready_counts=ready)
    sp.set_views(views, scene.camera_pos)
    for _ in range(3):
        sp.run()
    steady_launches = sp.last_launch_count()
    steady = float(np.median([timed(sp.run) for _ in range(max(a.reps, 5))]))
    print(f"steady frame: {steady:.3f} ms, {steady_launches} launches", flush=True)

    results = {"gpu": info, "n": a.n, "steady_frame_ms": steady, "cases": []}
    for frac in (0.001, 0.01, 0.1):
        count = int(occ * frac)
        for case in ("flags", "grow"):
            upd_ms, frame_ms, launches = [], [], []
            for _ in range(a.reps):
                slots = rng.choice(occ, size=count, replace=False).astype(np.uint32)
                if case == "flags":
                    m["isEnabled"][slots] ^= 1
                    m["isVisible"][slots] = rng.integers(0, 2, count).astype(np.uint8)
                    ready[slots] = rng.integers(0, 3, count).astype(np.uint8)
                else:
                    m["aabbMin"][slots, :3] *= np.float32(1.25)
                    m["aabbMax"][slots, :3] *= np.float32(1.25)
                upd_ms.append(timed(lambda: sp.update_mesh_pool_indexed(0, m, stride, slots, occ, ready)))
                frame_ms.append(timed(sp.run))
                launches.append(sp.last_launch_count())
            row = {"fraction": frac, "slots": count, "case": case, "update_ms": float(np.median(upd_ms)),
                   "next_frame_ms": float(np.median(frame_ms)), "launches_equal_steady": all(n == steady_launches for n in launches)}
            results["cases"].append(row)
            print(json.dumps(row), flush=True)

    restage_ms, frame_ms = [], []
    for _ in range(a.reps):
        restage_ms.append(timed(lambda: sp.set_mesh_pool(0, scene.pools[0].render_type, m, stride, occ, occ, ready_counts=ready)))
        frame_ms.append(timed(sp.run))
    row = {"case": "gsp_set_mesh_pool restage", "slots": occ, "update_ms": float(np.median(restage_ms)),
           "next_frame_ms": float(np.median(frame_ms)), "launches": sp.last_launch_count()}
    results["cases"].append(row)
    print(json.dumps(row), flush=True)

    # the updated context's lists against a context freshly staged from the same bytes (after one more scattered update)
    slots = rng.choice(occ, size=occ // 100, replace=False).astype(np.uint32)
    m["isEnabled"][slots] ^= 1
    m["aabbMax"][slots, :3] *= np.float32(2.0)
    sp.update_mesh_pool_indexed(0, m, stride, slots, occ, ready)
    sp.run()
    fresh = ScenePrep(0)
    fresh.set_transforms(t, 80, t.size)
    fresh.set_pool_count(1)
    fresh.set_mesh_pool(0, scene.pools[0].render_type, m, stride, occ, occ, ready_counts=ready)
    fresh.set_views(views, scene.camera_pos)
    fresh.run()
    same = all_lists(sp, views) == all_lists(fresh, views)
    results["lists_equal_fresh_staging"] = same
    print(f"lists equal a fresh staging: {same}", flush=True)
    fresh.close(); sp.close()
    for arr in (t, m, ready):
        unpin_host(arr)
    if a.json:
        with open(a.json, "w") as f:
            json.dump(results, f, indent=1)
    if not same:
        sys.exit(1)


if __name__ == "__main__":
    main()
